// Streaming fingerprinting (sia_stream_*, include/sia_b200.h): S independent streams on one context, each fed
// block by block, emitting every hash as soon as no later sample can change it.  The concatenated output of a stream
// equals sia_fingerprint_batch on its whole PCM (the reference's list order, __init__.py:198-208).
//
// Per stream, in HBM, two copies (the push writes the other copy and the host flips to it only when the push
// succeeded, so a failed push leaves every stream as it was):
//   tail   the samples after the next frame start (< 4096)
//   rows   the last min(2*nbhd, F) float32 dB rows: nbhd rows of context + nbhd rows whose peaks are not final
//   peaks  the non-final suffix of the peak list (< fan_value peaks)
// The host mirrors sample / frame / carried-peak counts, so a push is planned without reading the device.
//
// One push, chunk by chunk (streams whose carried + new rows fit the context workspace):
//   stage    tail + block -> 8-sample aligned staging PCM
//   K1       stft_db_kernel on the staged PCM: the new frames only, into the stream handle's row buffer
//   assemble carried rows + new rows -> the chunk spectrogram (one segment per stream)
//   K2       the bitmap kernels unchanged; rowcount / extract keep the rows of each stream's emit window
//            (H_prev, H] only and shift t to the stream's frame index
//   splice   carried peaks in front of each stream's new peaks
//   K3       pair counts with the finality rule (non-final anchors count 0), scan, pairs_sha1 unchanged
//   commit   new tail, rows and peak suffix -> the other state copy
// Finality: with F complete frames, H = F - 1 - nbhd is the last row whose whole neighbourhood is known; peaks in
// rows <= H are final; anchor i of the known peaks p_0..p_{n-1} is final iff i + fan_value - 1 < n or
// t_i <= H - MAX_HASH_TIME_DELTA (no later peak can be one of its partners).  At the end of a stream everything is.
#include "ctx.cuh"

#include <algorithm>
#include <climits>
#include <vector>

namespace sia {
namespace {

constexpr int kRowVec = SIA_F_STRIDE / 4;   // float4 per spectrogram row
constexpr int kTailCap = SIA_NFFT;          // tail slot (samples) per stream
constexpr int kPeakCap = 64;                // peak slots per stream (fan_value - 1 <= 63 are carried)

inline int64_t complete_frames(int64_t n, int hop) { return n >= SIA_NFFT ? 1 + (n - SIA_NFFT) / hop : 0; }

// per-chunk metadata (nb streams); every array lives in d_meta
struct StreamMeta {
  enum { kPerStream = 14, kPrefix = 6 };
  int64_t *st_start, *st_len;        // staged PCM of the stream (samples)
  int64_t *emit_lo, *emit_hi;        // segment-local rows whose peaks are emitted
  int64_t *t_base, *peak_off;        // frame index of the segment's first row; new peaks' offset (= cpre[b+1])
  int64_t *final_t;                  // anchors with t <= final_t are final
  int64_t *sid, *f_old, *r_old, *n_new, *r_new, *tail_new, *end;    // stream index, frame counts, next state
  int64_t *fs1, *fs2, *tt2, *cpre, *peak_starts, *hash_starts;   // [nb+1] each
  static size_t size(int nb) { return (size_t)nb * kPerStream + (size_t)kPrefix * (nb + 1); }
  StreamMeta(int64_t *base, int nb) {
    int64_t **per[kPerStream] = {&st_start, &st_len, &emit_lo, &emit_hi, &t_base, &peak_off, &final_t, &sid,
                                 &f_old, &r_old, &n_new, &r_new, &tail_new, &end};
    for (int i = 0; i < kPerStream; ++i) *per[i] = base + (size_t)i * nb;
    int64_t *q = base + (size_t)kPerStream * nb;
    int64_t **pre[kPrefix] = {&fs1, &fs2, &tt2, &cpre, &peak_starts, &hash_starts};
    for (int i = 0; i < kPrefix; ++i) *pre[i] = q + (size_t)i * (nb + 1);
  }
};

struct StreamChunk {
  int b0, b1;
  int64_t new_rows, rows, ttiles;
  size_t meta_off;
};

// tail + block -> staging; one CTA per stream
__global__ void __launch_bounds__(256)
stage_pcm_kernel(const int16_t *__restrict__ pcm, const int64_t *__restrict__ block_start, const int16_t *__restrict__ tails,
                 StreamMeta m, int16_t *__restrict__ stage) {
  const int b = blockIdx.x;
  const int64_t len = m.st_len[b];
  const int64_t tail = m.st_len[b] - (block_start[2 * b + 1]);
  const int64_t bs = block_start[2 * b];
  const int16_t *tl = tails + m.sid[b] * kTailCap;
  int16_t *dst = stage + m.st_start[b];
  for (int64_t i = threadIdx.x; i < len; i += blockDim.x) dst[i] = i < tail ? tl[i] : pcm[bs + i - tail];
}

// carried rows (state) + new rows (K1 output) -> the chunk spectrogram; one CTA per row
__global__ void __launch_bounds__(256)
assemble_rows_kernel(StreamMeta m, int nb, const float4 *__restrict__ rows_cur, int r2, const float4 *__restrict__ k1_rows,
                     float4 *__restrict__ spec) {
  const int64_t total = m.fs2[nb];
  for (int64_t g = blockIdx.x; g < total; g += gridDim.x) {
    const int b = find_segment(m.fs2, nb, g);
    const int64_t r = g - m.fs2[b];
    const float4 *src = r < m.r_old[b] ? rows_cur + ((size_t)m.sid[b] * r2 + r) * kRowVec
                                       : k1_rows + (size_t)(m.fs1[b] + r - m.r_old[b]) * kRowVec;
    float4 *dst = spec + (size_t)g * kRowVec;
    for (int i = threadIdx.x; i < kRowVec; i += blockDim.x) dst[i] = src[i];
  }
}

// per stream: start of its peak list (carried first, then the new peaks extract placed behind them) and the carried
// peaks themselves; one warp per stream (+ one for the end offset)
__global__ void __launch_bounds__(256)
splice_peaks_kernel(StreamMeta m, int nb, const int64_t *__restrict__ row_off, const int32_t *__restrict__ pk_t_cur,
                    const int32_t *__restrict__ pk_f_cur, int32_t *__restrict__ peak_t, int32_t *__restrict__ peak_f,
                    int64_t cap, int32_t *__restrict__ status) {
  const int lane = threadIdx.x & 31;
  const int64_t b = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (b > nb) return;
  const int64_t p = row_off[m.fs2[b]] + m.cpre[b];
  if (lane == 0) {
    m.peak_starts[b] = min(p, cap);
    if (b == nb && p > cap) atomicOr(status, 1);
  }
  if (b == nb) return;
  const int64_t n = m.cpre[b + 1] - m.cpre[b];
  const int64_t s = m.sid[b] * kPeakCap;
  for (int64_t j = lane; j < n; j += 32) {
    if (p + j < cap) { peak_t[p + j] = pk_t_cur[s + j]; peak_f[p + j] = pk_f_cur[s + j]; }
    else atomicOr(status, 1);
  }
}

__global__ void advance_base_kernel(int64_t *hash_base, const int64_t *end) { *hash_base = *end; }

// the stream's next state -> the other copy; one CTA per stream
__global__ void __launch_bounds__(256)
commit_kernel(StreamMeta m, int fan_value, int r2, const int32_t *__restrict__ peak_t, const int32_t *__restrict__ peak_f,
              const int16_t *__restrict__ stage, const float4 *__restrict__ k1_rows, const float4 *__restrict__ rows_cur,
              float4 *__restrict__ rows_nxt, int32_t *__restrict__ pk_t_nxt, int32_t *__restrict__ pk_f_nxt,
              int16_t *__restrict__ tails_nxt, int32_t *__restrict__ n_carried) {
  __shared__ int64_t s_first;
  const int b = blockIdx.x;
  const int64_t sid = m.sid[b];
  const int64_t p0 = m.peak_starts[b], p1 = m.peak_starts[b + 1];
  if (threadIdx.x == 0) {
    int64_t k = p1 - p0;   // first non-final peak: all final at the end
    if (!m.end[b]) {
      int64_t lo = p0, hi = p1;   // peaks with t <= final_t form a prefix (t is non-decreasing)
      while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (peak_t[mid] <= m.final_t[b]) lo = mid + 1; else hi = mid;
      }
      k = max(lo - p0, p1 - p0 - (fan_value - 1));
      k = max(k, (int64_t)0);
    }
    s_first = p0 + k;
    n_carried[sid] = (int32_t)(p1 - p0 - k);
  }
  __syncthreads();
  for (int64_t i = s_first + threadIdx.x; i < p1; i += blockDim.x) {
    pk_t_nxt[sid * kPeakCap + (i - s_first)] = peak_t[i];
    pk_f_nxt[sid * kPeakCap + (i - s_first)] = peak_f[i];
  }
  // rows: absolute rows [f_new - r_new, f_new); old rows [f_old - r_old, f_old) sit in the state, new ones in k1_rows
  const int64_t f_old = m.f_old[b], f_new = f_old + m.n_new[b], r_new = m.r_new[b];
  for (int64_t j = 0; j < r_new; ++j) {
    const int64_t a = f_new - r_new + j;
    const float4 *src = a < f_old ? rows_cur + ((size_t)sid * r2 + (a - (f_old - m.r_old[b]))) * kRowVec
                                  : k1_rows + (size_t)(m.fs1[b] + a - f_old) * kRowVec;
    float4 *dst = rows_nxt + ((size_t)sid * r2 + j) * kRowVec;
    for (int i = threadIdx.x; i < kRowVec; i += blockDim.x) dst[i] = src[i];
  }
  // tail: staged samples from the next frame start on
  const int64_t tn = m.tail_new[b];
  const int16_t *ts = stage + m.st_start[b] + m.st_len[b] - tn;
  for (int64_t i = threadIdx.x; i < tn; i += blockDim.x) tails_nxt[sid * kTailCap + i] = ts[i];
}

}  // namespace
}  // namespace sia

using namespace sia;

struct sia_stream {
  sia_ctx *c = nullptr;
  int32_t n = 0;
  sia_fp_params p{};
  int hop = 0;                         // frame k starts at sample k * hop (fp_hop of p)
  int r2 = 0;                          // 2 * nbhd carried rows
  int cur = 0;                         // state copy of the last successful push
  int16_t *tails[2] = {nullptr, nullptr};
  float *rows[2] = {nullptr, nullptr};
  int32_t *pk_t[2] = {nullptr, nullptr}, *pk_f[2] = {nullptr, nullptr};
  int32_t *n_carried = nullptr;        // [n] carried peaks after the push (read back)
  float *k1_rows = nullptr;            // [max_frames][F_STRIDE] new rows of a chunk
  int64_t *d_blocks = nullptr;         // [n][2] (block start, block length)
  int16_t *stage = nullptr;
  int64_t stage_cap = 0;
  std::vector<int64_t> L, F, npk;      // host mirror: samples, complete frames, carried peaks
};

extern "C" {

int sia_stream_destroy(sia_stream *st) {
  SIA_REQUIRE(st != nullptr, SIA_E_INVALID, "stream handle is NULL");
  cudaSetDevice(st->c->device);
  cudaDeviceSynchronize();
  void *ptrs[] = {st->tails[0], st->tails[1], st->rows[0], st->rows[1], st->pk_t[0], st->pk_t[1], st->pk_f[0],
                  st->pk_f[1], st->n_carried, st->k1_rows, st->d_blocks, st->stage};
  for (void *q : ptrs) if (q) cudaFree(q);
  delete st;
  return SIA_OK;
}

int sia_stream_create(sia_ctx *c, int32_t n_streams, const sia_fp_params *p, sia_stream **out) {
  SIA_REQUIRE(out != nullptr, SIA_E_INVALID, "out is NULL");
  *out = nullptr;
  SIA_REQUIRE(c != nullptr, SIA_E_INVALID, "ctx is NULL");
  SIA_REQUIRE(n_streams >= 1, SIA_E_INVALID, "n_streams must be >= 1");
  int rc = check_params(p);
  if (rc) return rc;
  SIA_CUDA(cudaSetDevice(c->device));
  sia_stream *st = new (std::nothrow) sia_stream();
  SIA_REQUIRE(st != nullptr, SIA_E_NOMEM, "out of host memory");
  st->c = c; st->n = n_streams; st->p = *p; st->hop = fp_hop(p); st->r2 = 2 * p->nbhd;
  st->L.assign(n_streams, 0); st->F.assign(n_streams, 0); st->npk.assign(n_streams, 0);
  const size_t S = (size_t)n_streams;
  auto alloc = [&](void **q, size_t bytes) -> int {
    cudaError_t e = cudaMalloc(q, bytes);
    if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc (stream state)", __FILE__, __LINE__);
    return SIA_OK;
  };
  for (int i = 0; i < 2 && !rc; ++i) {
    if (!rc) rc = alloc((void **)&st->tails[i], S * kTailCap * sizeof(int16_t));
    if (!rc) rc = alloc((void **)&st->rows[i], S * st->r2 * SIA_F_STRIDE * sizeof(float));
    if (!rc) rc = alloc((void **)&st->pk_t[i], S * kPeakCap * sizeof(int32_t));
    if (!rc) rc = alloc((void **)&st->pk_f[i], S * kPeakCap * sizeof(int32_t));
  }
  if (!rc) rc = alloc((void **)&st->n_carried, S * sizeof(int32_t));
  if (!rc) rc = alloc((void **)&st->k1_rows, (size_t)c->max_frames * SIA_F_STRIDE * sizeof(float));
  if (!rc) rc = alloc((void **)&st->d_blocks, S * 2 * sizeof(int64_t));
  if (rc) { sia_stream_destroy(st); return rc; }
  *out = st;
  return SIA_OK;
}

int sia_stream_push(sia_stream *st, const int16_t *d_pcm, const int64_t *h_block_starts, const int64_t *h_block_len,
                    const uint8_t *h_end, uint8_t *d_hash, int32_t *d_t1, int64_t cap_hashes,
                    int64_t *h_stream_hash_starts, int64_t *h_total, void *stream) {
  SIA_REQUIRE(st && h_block_starts && h_block_len && h_total, SIA_E_INVALID, "NULL argument");
  SIA_REQUIRE(cap_hashes >= 0, SIA_E_INVALID, "cap_hashes < 0");
  SIA_REQUIRE(cap_hashes == 0 || (d_hash && d_t1), SIA_E_INVALID, "NULL device output buffer");
  const int S = st->n;
  bool any_pcm = false;
  for (int b = 0; b < S; ++b) {
    SIA_REQUIRE(h_block_len[b] >= 0, SIA_E_INVALID, "negative block length");
    SIA_REQUIRE(h_block_len[b] == 0 || h_block_starts[b] % 8 == 0, SIA_E_INVALID,
                "block starts must be multiples of 8 samples");
    any_pcm |= h_block_len[b] > 0;
  }
  SIA_REQUIRE(!any_pcm || d_pcm, SIA_E_INVALID, "d_pcm is NULL");
  sia_ctx *c = st->c;
  const sia_fp_params &p = st->p;
  const int nbhd = p.nbhd, hop = st->hop;
  SIA_CUDA(cudaSetDevice(c->device));
  cudaStream_t s = (cudaStream_t)stream;

  // ---- plan (host only) ----
  struct Plan { int64_t tail, st_start, st_len, f_new, n_new, r_old, r_new, tail_new, lo, hi, t_base, final_t; bool end; };
  std::vector<Plan> pl(S);
  int64_t stage_total = 0;
  for (int b = 0; b < S; ++b) {
    Plan &q = pl[b];
    const int64_t F = st->F[b], L = st->L[b];
    q.end = h_end && h_end[b];
    q.tail = L - F * hop;
    q.st_start = stage_total;
    q.st_len = q.tail + h_block_len[b];
    stage_total += (q.st_len + 7) / 8 * 8;
    const int64_t Ln = L + h_block_len[b];
    int64_t Fn = complete_frames(Ln, hop);
    if (q.end && Fn == 0) Fn = 1;       // short input: one zero-padded frame, like the batch path
    q.f_new = Fn;
    q.n_new = Fn - F;
    q.r_old = std::min<int64_t>(st->r2, F);
    q.r_new = q.end ? 0 : std::min<int64_t>(st->r2, Fn);
    q.tail_new = q.end ? 0 : q.st_len - q.n_new * hop;
    q.t_base = F - q.r_old;
    const int64_t h_old = F - 1 - nbhd, h_new = q.end ? Fn - 1 : Fn - 1 - nbhd;
    q.lo = std::max<int64_t>(h_old + 1, 0) - q.t_base;
    q.hi = std::max(q.lo, h_new + 1 - q.t_base);
    q.final_t = q.end ? INT_MAX : h_new - SIA_MAX_DT;
  }
  auto seg_rows = [&](const Plan &q) -> int64_t { return (q.n_new > 0 || q.end) ? q.r_old + q.n_new : 0; };
  std::vector<StreamChunk> chunks;
  size_t meta_total = 0;
  for (int b = 0; b < S;) {
    StreamChunk ch{b, b, 0, 0, 0, meta_total};
    while (ch.b1 < S) {
      const int64_t r = seg_rows(pl[ch.b1]);
      if (r > c->max_frames) {
        char buf[256];
        snprintf(buf, sizeof buf, "stream %d needs %lld spectrogram rows in this push (carried + new frames); the context "
                 "workspace holds %lld: push smaller blocks or raise max_chunk_frames", ch.b1, (long long)r,
                 (long long)c->max_frames);
        set_error(buf);
        return SIA_E_CAPACITY;
      }
      if (ch.rows + r > c->max_frames) break;
      ch.rows += r;
      ch.new_rows += seg_rows(pl[ch.b1]) ? pl[ch.b1].n_new : 0;
      ch.ttiles += ceil_div(r, kPeakTileT);
      ++ch.b1;
    }
    meta_total += StreamMeta::size(ch.b1 - ch.b0);
    chunks.push_back(ch);
    b = ch.b1;
  }
  int rc;
  if ((rc = ensure_meta(c, meta_total))) return rc;
  const size_t blocks_off = meta_total, tail_off = meta_total + 2 * (size_t)S;
  if ((rc = ensure_pinned(c, tail_off + 4 + (size_t)S))) return rc;
  if (stage_total > st->stage_cap) {
    if (st->stage) cudaFree(st->stage);
    st->stage = nullptr;
    st->stage_cap = 0;
    const int64_t cap = std::max<int64_t>(stage_total + stage_total / 4, 1 << 16);
    SIA_CUDA(cudaMalloc(&st->stage, (size_t)cap * sizeof(int16_t)));
    st->stage_cap = cap;
  }
  int64_t *hm_all = c->h_pinned;
  for (const StreamChunk &ch : chunks) {
    const int nb = ch.b1 - ch.b0;
    StreamMeta m(hm_all + ch.meta_off, nb);
    int64_t fs1 = 0, fs2 = 0, tt2 = 0, cpre = 0;
    for (int i = 0; i < nb; ++i) {
      const int b = ch.b0 + i;
      const Plan &q = pl[b];
      const int64_t rows = seg_rows(q);
      m.fs1[i] = fs1; m.fs2[i] = fs2; m.tt2[i] = tt2; m.cpre[i] = cpre;
      fs1 += rows ? q.n_new : 0; fs2 += rows; tt2 += ceil_div(rows, kPeakTileT); cpre += st->npk[b];
      m.st_start[i] = q.st_start; m.st_len[i] = q.st_len;
      m.emit_lo[i] = rows ? q.lo : 0; m.emit_hi[i] = rows ? q.hi : 0;
      m.t_base[i] = q.t_base; m.peak_off[i] = cpre; m.final_t[i] = q.final_t;
      m.sid[i] = b; m.f_old[i] = st->F[b]; m.r_old[i] = q.r_old; m.n_new[i] = q.n_new; m.r_new[i] = q.r_new;
      m.tail_new[i] = q.tail_new; m.end[i] = q.end;
      m.peak_starts[i] = m.hash_starts[i] = 0;
    }
    m.fs1[nb] = fs1; m.fs2[nb] = fs2; m.tt2[nb] = tt2; m.cpre[nb] = cpre;
    m.peak_starts[nb] = m.hash_starts[nb] = 0;
  }
  for (int b = 0; b < S; ++b) {
    hm_all[blocks_off + 2 * b] = h_block_starts[b];
    hm_all[blocks_off + 2 * b + 1] = h_block_len[b];
  }

  // ---- device pass ----
  SIA_CUDA(cudaMemcpyAsync(c->d_meta, hm_all, meta_total * sizeof(int64_t), cudaMemcpyHostToDevice, s));
  SIA_CUDA(cudaMemcpyAsync(st->d_blocks, hm_all + blocks_off, 2 * (size_t)S * sizeof(int64_t), cudaMemcpyHostToDevice, s));
  SIA_CUDA(cudaMemsetAsync(c->status, 0, sizeof(int32_t), s));
  SIA_CUDA(cudaMemsetAsync(c->hash_base, 0, sizeof(int64_t), s));
  const int cur = st->cur, nxt = cur ^ 1;
  const float4 *rows_cur = reinterpret_cast<const float4 *>(st->rows[cur]);
  const float4 *k1 = reinterpret_cast<const float4 *>(st->k1_rows);
  for (const StreamChunk &ch : chunks) {
    const int nb = ch.b1 - ch.b0;
    StreamMeta m(c->d_meta + ch.meta_off, nb);
    {
      Timer t(c, s, T_STREAM, 1);
      stage_pcm_kernel<<<nb, 256, 0, s>>>(d_pcm, st->d_blocks + 2 * (size_t)ch.b0, st->tails[cur], m, st->stage);
      SIA_CHECK_LAUNCH();
    }
    bool striped = false;
    if (ch.rows > 0) {
      StftLaunch a;
      a.d_pcm = st->stage; a.d_track_starts = m.st_start; a.d_track_len = m.st_len; a.d_frame_starts = m.fs1;
      a.n_tracks = nb; a.total_frames = ch.new_rows; a.d_spec = st->k1_rows; a.out_type = SIA_F32;
      a.frames_per_cta = 8; a.compute = p.compute; a.Fs = p.Fs; a.hop = hop;
      if (ch.new_rows > 0) {
        Timer t(c, s, T_STFT, 1);
        if ((rc = stft_db_launch(a, c->tf, c->td, s))) return rc;
      }
      {
        Timer t(c, s, T_STREAM, 1);
        assemble_rows_kernel<<<(unsigned)std::min<int64_t>(ch.rows, kNumSMs * 32), 256, 0, s>>>(
            m, nb, rows_cur, st->r2, k1, reinterpret_cast<float4 *>(c->spec));
        SIA_CHECK_LAUNCH();
      }
      PeaksLaunch pk;
      pk.d_spec = c->spec; pk.in_type = SIA_F32; pk.d_frame_starts = m.fs2; pk.d_ttile_starts = m.tt2;
      pk.n_tracks = nb; pk.total_frames = ch.rows; pk.total_ttiles = ch.ttiles; pk.amp_min = p.amp_min;
      pk.connectivity = p.connectivity; pk.nbhd = p.nbhd; pk.d_bitmap = c->bitmap;
      {
        Timer t(c, s, T_PEAKS, 1);
        if ((rc = peaks_bitmap_launch(pk, s, &striped))) return rc;
      }
      const PeakWindow win{m.fs2, m.emit_lo, m.emit_hi, m.t_base, m.peak_off, nb};
      {
        Timer t(c, s, T_COMPACT, 1);
        if ((rc = peaks_rowcount_launch(c->bitmap, striped, ch.rows, c->row_count, s, &win))) return rc;
      }
      {
        Timer t(c, s, T_SCAN, 3);
        if ((rc = exclusive_scan_u32(c->row_count, c->row_off, ch.rows, c->scan_tmp, s))) return rc;
      }
      {
        Timer t(c, s, T_COMPACT, 1);
        if ((rc = peaks_extract_launch(c->bitmap, striped, c->row_off, m.fs2, nb, ch.rows, 0, c->peak_t, c->peak_f,
                                       c->cap_peaks, nullptr, c->status, s, &win)))
          return rc;
      }
    } else {
      SIA_CUDA(cudaMemsetAsync(c->row_off, 0, sizeof(int64_t), s));
    }
    {
      Timer t(c, s, T_STREAM, 1);
      splice_peaks_kernel<<<(unsigned)ceil_div((int64_t)(nb + 1) * 32, 256), 256, 0, s>>>(
          m, nb, c->row_off, st->pk_t[cur], st->pk_f[cur], c->peak_t, c->peak_f, c->cap_peaks, c->status);
      SIA_CHECK_LAUNCH();
    }
    {
      Timer t(c, s, T_PAIRS, 1);
      if ((rc = pairs_count_launch(c->peak_t, m.peak_starts, nb, c->cap_peaks, p.fan_value, c->pair_count, s, m.final_t)))
        return rc;
    }
    {
      Timer t(c, s, T_SCAN, 3);
      if ((rc = exclusive_scan_u32_dyn(c->pair_count, c->pair_off, m.peak_starts + nb, c->cap_peaks, c->scan_tmp, s)))
        return rc;
    }
    {
      Timer t(c, s, T_PAIRS, 3);
      if ((rc = pairs_sha1_launch(c->peak_t, c->peak_f, m.peak_starts, nb, c->cap_peaks, p.fan_value, c->pair_count,
                                  c->pair_off, 0, c->hash_base, c->digest_table, d_hash, d_t1, cap_hashes, m.hash_starts,
                                  c->status, s)))
        return rc;
      advance_base_kernel<<<1, 1, 0, s>>>(c->hash_base, m.hash_starts + nb);
      SIA_CHECK_LAUNCH();
    }
    {
      Timer t(c, s, T_STREAM, 1);
      commit_kernel<<<nb, 256, 0, s>>>(m, p.fan_value, st->r2, c->peak_t, c->peak_f, st->stage, k1, rows_cur,
                                       reinterpret_cast<float4 *>(st->rows[nxt]), st->pk_t[nxt], st->pk_f[nxt],
                                       st->tails[nxt], st->n_carried);
      SIA_CHECK_LAUNCH();
    }
  }
  // results: per-stream offsets, total, status, carried peak counts — one synchronisation
  int64_t *back = c->h_pinned + tail_off;
  int32_t *h_nc = reinterpret_cast<int32_t *>(back + 4);
  SIA_CUDA(cudaMemcpyAsync(c->h_pinned, c->d_meta, meta_total * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
  SIA_CUDA(cudaMemcpyAsync(back, c->hash_base, sizeof(int64_t), cudaMemcpyDeviceToHost, s));
  SIA_CUDA(cudaMemcpyAsync(back + 1, c->status, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
  SIA_CUDA(cudaMemcpyAsync(h_nc, st->n_carried, (size_t)S * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
  SIA_CUDA(cudaStreamSynchronize(s));
  const int64_t total = back[0];
  const int32_t status = *reinterpret_cast<int32_t *>(back + 1);
  *h_total = total;
  if (h_stream_hash_starts) {
    for (const StreamChunk &ch : chunks) {
      const int nb = ch.b1 - ch.b0;
      StreamMeta m(c->h_pinned + ch.meta_off, nb);
      for (int i = 0; i < nb; ++i) h_stream_hash_starts[ch.b0 + i] = m.hash_starts[i];
    }
    h_stream_hash_starts[S] = total;
  }
  if (status & 1) {
    set_error("peak workspace overflow: more than SIA_PEAKS_PER_FRAME_CAP (default 32) peaks per frame on average; "
              "set the environment variable higher and recreate the context");
    return SIA_E_CAPACITY;
  }
  if ((status & 2) || total > cap_hashes) {
    set_error("hash output capacity exceeded; *h_total holds the required number of rows");
    return SIA_E_CAPACITY;
  }
  // success: the pushed state becomes the current one
  st->cur = nxt;
  for (int b = 0; b < S; ++b) {
    const Plan &q = pl[b];
    if (q.end) { st->L[b] = 0; st->F[b] = 0; st->npk[b] = 0; continue; }
    st->L[b] += h_block_len[b];
    st->F[b] = q.f_new;
    st->npk[b] = h_nc[b];
  }
  return SIA_OK;
}

}  // extern "C"
