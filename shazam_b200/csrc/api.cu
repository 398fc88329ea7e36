// C ABI of the fingerprint path (include/sia_b200.h): context, workspaces, chunking of a
// batch of tracks through K1 -> K2 -> K3, and the pinned-host pipeline
// (H2D | kernels | D2H on three streams).  This is the native runtime behind
// fingerprint()/_fingerprint_worker (__init__.py:212-284): the reference fans tracks out
// over a multiprocessing.Pool; here a batch is one call and the chunk loop is the pool.
#include "ctx.cuh"

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <vector>

namespace sia {

static thread_local std::string g_last_error;
void set_error(const std::string &msg) { g_last_error = msg; }
int cuda_fail(cudaError_t e, const char *what, const char *file, int line) {
  char buf[512];
  snprintf(buf, sizeof buf, "CUDA error %d (%s) at %s:%d: %s", (int)e, cudaGetErrorString(e), file, line, what);
  g_last_error = buf;
  return SIA_E_CUDA;
}

}  // namespace sia

using namespace sia;

namespace sia {

int check_params(const sia_fp_params *p) {
  SIA_REQUIRE(p != nullptr, SIA_E_INVALID, "params is NULL");
  SIA_REQUIRE(p->wsize == SIA_NFFT, SIA_E_UNSUPPORTED, "only wsize=4096 (DEFAULT_WINDOW_SIZE) is implemented");
  // noverlap = int(4096 * wratio) must be 0..4095; tested on the product before the conversion to an integer
  const double noverlap = SIA_NFFT * p->wratio;
  SIA_REQUIRE(!(noverlap != noverlap) && noverlap < SIA_NFFT, SIA_E_INVALID,
              "wratio must give noverlap = int(4096 * wratio) <= 4095 (a hop of at least one sample)");
  SIA_REQUIRE(noverlap > -1.0, SIA_E_UNSUPPORTED,
              "wratio < 0 (noverlap < 0: gaps between frames) is not implemented");
  SIA_REQUIRE(p->Fs > 0, SIA_E_INVALID, "Fs must be positive");
  SIA_REQUIRE(p->fan_value >= 1 && p->fan_value <= 64, SIA_E_INVALID, "fan_value must be in 1..64");
  SIA_REQUIRE(p->connectivity == 1 || p->connectivity == 2, SIA_E_INVALID, "connectivity must be 1 or 2");
  SIA_REQUIRE(p->nbhd >= 1 && p->nbhd <= SIA_MAX_NBHD, SIA_E_INVALID, "nbhd must be in 1..64");
  SIA_REQUIRE(p->compute == SIA_F32 || p->compute == SIA_F64, SIA_E_INVALID, "compute must be SIA_F32 or SIA_F64");
  return SIA_OK;
}

int ensure_meta(sia_ctx *c, size_t n_i64) {
  if (n_i64 <= c->d_meta_cap) return SIA_OK;
  if (c->d_meta) cudaFree(c->d_meta);
  c->d_meta = nullptr;
  c->d_meta_cap = 0;
  size_t cap = std::max<size_t>(n_i64, 4096);
  SIA_CUDA(cudaMalloc(&c->d_meta, cap * sizeof(int64_t)));
  c->d_meta_cap = cap;
  return SIA_OK;
}

int ensure_pinned(sia_ctx *c, size_t n_i64) {
  if (n_i64 <= c->h_pinned_cap) return SIA_OK;
  if (c->h_pinned) cudaFreeHost(c->h_pinned);
  c->h_pinned = nullptr;
  c->h_pinned_cap = 0;
  size_t cap = std::max<size_t>(n_i64, 4096);
  SIA_CUDA(cudaMallocHost(&c->h_pinned, cap * sizeof(int64_t)));
  c->h_pinned_cap = cap;
  return SIA_OK;
}

}  // namespace sia

namespace {

void collect_timing(sia_ctx *c) {
  for (auto &sp : c->spans) {
    float ms = 0;
    if (cudaEventElapsedTime(&ms, sp.a, sp.b) == cudaSuccess) c->ms[sp.cat] += ms;
    c->ev_pool.push_back(sp.a);
    c->ev_pool.push_back(sp.b);
  }
  c->spans.clear();
}

// One chunk = tracks [b0, b1) whose frames fit the workspace.
struct Chunk {
  int b0, b1;
  int64_t frames, ttiles;
  size_t meta_off;    // offset (int64 units) of this chunk's metadata block in d_meta
};

// metadata block layout per chunk (nb = b1-b0): track_starts[nb] | track_len[nb] | frame_starts[nb+1] |
// ttile_starts[nb+1] | track_peak_starts[nb+1] | track_hash_starts[nb+1]
struct MetaView {
  int64_t *track_starts, *track_len, *frame_starts, *ttile_starts, *track_peak_starts, *track_hash_starts;
  static size_t size(int nb) { return (size_t)nb * 2 + 4 * ((size_t)nb + 1); }
  MetaView(int64_t *base, int nb) {
    track_starts = base; track_len = base + nb; frame_starts = base + 2 * (size_t)nb;
    ttile_starts = frame_starts + nb + 1; track_peak_starts = ttile_starts + nb + 1;
    track_hash_starts = track_peak_starts + nb + 1;
  }
};

// max_samples > 0 additionally bounds the (8-sample padded) PCM of a chunk — the staging buffer of the
// host pipeline.
int plan_chunks(sia_ctx *c, const sia_fp_params *p, const int64_t *h_len, int n_tracks, int64_t max_samples,
                std::vector<Chunk> &chunks) {
  chunks.clear();
  size_t meta = 0;
  int b = 0;
  while (b < n_tracks) {
    Chunk ch{b, b, 0, 0, meta};
    int64_t samples = 0;
    while (ch.b1 < n_tracks) {
      const int64_t fr = fp_frames(p, h_len[ch.b1]);
      if (fr > c->max_frames) {
        char buf[256];
        snprintf(buf, sizeof buf, "track %d has %lld frames; the context workspace holds %lld (raise max_chunk_frames, "
                 "or fingerprint it block by block with sia_stream_push)",
                 ch.b1, (long long)fr, (long long)c->max_frames);
        set_error(buf);
        return SIA_E_CAPACITY;
      }
      if (ch.frames + fr > c->max_frames) break;
      const int64_t padded = (h_len[ch.b1] + 7) / 8 * 8 + 8;
      if (max_samples > 0 && ch.b1 > ch.b0 && samples + padded > max_samples) break;
      samples += padded;
      ch.frames += fr;
      ch.ttiles += ceil_div(fr, kPeakTileT);
      ++ch.b1;
    }
    meta += MetaView::size(ch.b1 - ch.b0);
    chunks.push_back(ch);
    b = ch.b1;
  }
  return SIA_OK;
}

// Fill the host copy of every chunk's metadata.  dev_starts[b] = sample offset of track b inside the
// device PCM buffer the chunk's kernels will read.
void fill_meta(const std::vector<Chunk> &chunks, const sia_fp_params *p, const int64_t *dev_starts, const int64_t *h_len,
               int64_t *h_meta) {
  for (const Chunk &ch : chunks) {
    const int nb = ch.b1 - ch.b0;
    MetaView m(h_meta + ch.meta_off, nb);
    int64_t fr = 0, tt = 0;
    for (int i = 0; i < nb; ++i) {
      m.track_starts[i] = dev_starts[ch.b0 + i];
      m.track_len[i] = h_len[ch.b0 + i];
      m.frame_starts[i] = fr;
      m.ttile_starts[i] = tt;
      const int64_t f = fp_frames(p, h_len[ch.b0 + i]);
      fr += f;
      tt += ceil_div(f, kPeakTileT);
    }
    m.frame_starts[nb] = fr;
    m.ttile_starts[nb] = tt;
    for (int i = 0; i <= nb; ++i) m.track_peak_starts[i] = m.track_hash_starts[i] = 0;
  }
}

int64_t env_i64(const char *name, int64_t dflt);

int run_stft(sia_ctx *c, const int16_t *d_pcm, const MetaView &m, int nb, int64_t frames, const sia_fp_params *p,
             void *d_spec, int out_type, cudaStream_t s) {
  StftLaunch a;
  a.d_pcm = d_pcm; a.d_track_starts = m.track_starts; a.d_track_len = m.track_len; a.d_frame_starts = m.frame_starts;
  a.n_tracks = nb; a.total_frames = frames; a.d_spec = d_spec; a.out_type = out_type;
  a.frames_per_cta = 8;      // frames per CTA run (K1's PCM cursor keeps a clamped 32-bit remainder: runs stay short)
  a.compute = p->compute; a.Fs = p->Fs; a.hop = fp_hop(p);
  Timer t(c, s, T_STFT, 1);
  return stft_db_launch(a, c->tf, c->td, s);
}

int run_peaks(sia_ctx *c, const void *d_spec, int in_type, const MetaView &m, int nb, int64_t frames, int64_t ttiles,
              const sia_fp_params *p, int32_t *d_peak_t, int32_t *d_peak_f, int64_t cap_peaks,
              int64_t *d_track_peak_starts, int32_t *d_status, cudaStream_t s) {
  int rc;
  bool striped = false;
  {
    PeaksLaunch a;
    a.d_spec = d_spec; a.in_type = in_type; a.d_frame_starts = m.frame_starts; a.d_ttile_starts = m.ttile_starts;
    a.n_tracks = nb; a.total_frames = frames; a.total_ttiles = ttiles; a.amp_min = p->amp_min;
    a.connectivity = p->connectivity; a.nbhd = p->nbhd; a.d_bitmap = c->bitmap;
    Timer t(c, s, T_PEAKS, 1);
    if ((rc = peaks_bitmap_launch(a, s, &striped))) return rc;
  }
  {
    Timer t(c, s, T_COMPACT, 1);
    if ((rc = peaks_rowcount_launch(c->bitmap, striped, frames, c->row_count, s))) return rc;
  }
  {
    Timer t(c, s, T_SCAN, 3);
    if ((rc = exclusive_scan_u32(c->row_count, c->row_off, frames, c->scan_tmp, s))) return rc;
  }
  {
    Timer t(c, s, T_COMPACT, 1);
    if ((rc = peaks_extract_launch(c->bitmap, striped, c->row_off, m.frame_starts, nb, frames, 0, d_peak_t, d_peak_f, cap_peaks,
                                   d_track_peak_starts, d_status, s)))
      return rc;
  }
  return SIA_OK;
}

int run_pairs(sia_ctx *c, const int32_t *d_peak_t, const int32_t *d_peak_f, const int64_t *d_track_peak_starts, int nb,
              int64_t n_peaks_max, int fan_value, int64_t hash_base_static, const int64_t *d_hash_base,
              uint8_t *d_hash, int32_t *d_t1, int64_t cap_hashes, int64_t *d_track_hash_starts, int32_t *d_status,
              cudaStream_t s) {
  int rc;
  {
    Timer t(c, s, T_PAIRS, 1);
    if ((rc = pairs_count_launch(d_peak_t, d_track_peak_starts, nb, n_peaks_max, fan_value, c->pair_count, s))) return rc;
  }
  {
    Timer t(c, s, T_SCAN, 3);
    if ((rc = exclusive_scan_u32_dyn(c->pair_count, c->pair_off, d_track_peak_starts + nb, n_peaks_max, c->scan_tmp, s)))
      return rc;
  }
  {
    Timer t(c, s, T_PAIRS, 2);
    if ((rc = pairs_sha1_launch(d_peak_t, d_peak_f, d_track_peak_starts, nb, n_peaks_max, fan_value, c->pair_count,
                                c->pair_off, hash_base_static, d_hash_base, c->digest_table, d_hash, d_t1, cap_hashes,
                                d_track_hash_starts, d_status, s)))
      return rc;
  }
  return SIA_OK;
}

__global__ void advance_base_kernel(int64_t *hash_base, const int64_t *track_hash_starts_end, int64_t *chunk_count_out) {
  const int64_t end = *track_hash_starts_end;
  if (chunk_count_out) *chunk_count_out = end - *hash_base;
  *hash_base = end;
}

// K1..K3 for one chunk.  Digests go to d_hash/d_t1 at (*hash_base on the device) + local offset.
int run_chunk(sia_ctx *c, const int16_t *d_pcm, const Chunk &ch, const sia_fp_params *p, uint8_t *d_hash,
              int32_t *d_t1, int64_t cap_hashes, cudaStream_t s) {
  const int nb = ch.b1 - ch.b0;
  MetaView m(c->d_meta + ch.meta_off, nb);
  int rc;
  if ((rc = run_stft(c, d_pcm, m, nb, ch.frames, p, c->spec, SIA_F32, s))) return rc;
  if ((rc = run_peaks(c, c->spec, SIA_F32, m, nb, ch.frames, ch.ttiles, p, c->peak_t, c->peak_f, c->cap_peaks,
                      m.track_peak_starts, c->status, s)))
    return rc;
  if ((rc = run_pairs(c, c->peak_t, c->peak_f, m.track_peak_starts, nb, c->cap_peaks, p->fan_value, 0, c->hash_base,
                      d_hash, d_t1, cap_hashes, m.track_hash_starts, c->status, s)))
    return rc;
  advance_base_kernel<<<1, 1, 0, s>>>(c->hash_base, m.track_hash_starts + nb, nullptr);
  SIA_CHECK_LAUNCH();
  c->launches[T_PAIRS] += 1;
  return SIA_OK;
}

// ---- PCM de-interleave (read(), __init__.py:91-95) ---------------------------------------------------------
// stereo: one 16-byte load (4 frames) -> two 8-byte stores; other channel counts: scalar, coalesced on the reads
__global__ void __launch_bounds__(256)
deinterleave2_kernel(const int16_t *__restrict__ in, int64_t n_frames, int16_t *__restrict__ out, int64_t stride) {
  const int64_t nq = n_frames >> 2;                       // groups of 4 frames
  for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < nq; q += (int64_t)gridDim.x * blockDim.x) {
    const uint4 v = reinterpret_cast<const uint4 *>(in)[q];
    uint2 l, r;
    l.x = __byte_perm(v.x, v.y, 0x5410); r.x = __byte_perm(v.x, v.y, 0x7632);
    l.y = __byte_perm(v.z, v.w, 0x5410); r.y = __byte_perm(v.z, v.w, 0x7632);
    reinterpret_cast<uint2 *>(out)[q] = l;
    reinterpret_cast<uint2 *>(out + stride)[q] = r;
  }
  if (blockIdx.x == 0 && threadIdx.x < (n_frames & 3)) {   // tail frames
    const int64_t i = (nq << 2) + threadIdx.x;
    out[i] = in[2 * i]; out[stride + i] = in[2 * i + 1];
  }
}
__global__ void __launch_bounds__(256)
deinterleave_kernel(const int16_t *__restrict__ in, int64_t n_frames, int n_channels, int16_t *__restrict__ out, int64_t stride) {
  const int64_t n = n_frames * n_channels;
  for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = k / n_channels;
    const int c = (int)(k - i * n_channels);
    out[c * stride + i] = in[k];
  }
}

int64_t env_i64(const char *name, int64_t dflt) {
  const char *v = getenv(name);
  if (!v || !*v) return dflt;
  return atoll(v);
}

}  // namespace

extern "C" {

const char *sia_last_error(void) { return g_last_error.c_str(); }
int sia_version(void) { return 100; }

void sia_fp_params_default(sia_fp_params *p) {
  if (!p) return;
  p->Fs = 44100.0; p->wsize = 4096; p->wratio = 0.5; p->fan_value = 5; p->amp_min = 10.0;
  p->connectivity = 2; p->nbhd = 10; p->compute = SIA_F64;
}

int sia_deinterleave_i16(const int16_t *d_in, int64_t n_frames, int32_t n_channels, int16_t *d_out, int64_t channel_stride,
                         void *stream) {
  SIA_REQUIRE(n_frames >= 0 && n_channels >= 1 && n_channels <= 64, SIA_E_INVALID, "deinterleave: bad sizes");
  SIA_REQUIRE(channel_stride >= n_frames, SIA_E_INVALID, "deinterleave: channel_stride < n_frames");
  if (n_frames == 0) return SIA_OK;
  SIA_REQUIRE(d_in && d_out, SIA_E_INVALID, "NULL argument");
  cudaStream_t s = (cudaStream_t)stream;
  const bool vec = n_channels == 2 && (reinterpret_cast<uintptr_t>(d_in) & 15) == 0 &&
                   (reinterpret_cast<uintptr_t>(d_out) & 7) == 0 && (channel_stride & 3) == 0;
  if (vec) {
    const unsigned blocks = (unsigned)std::min<int64_t>(ceil_div(std::max<int64_t>(n_frames >> 2, 1), 256), kNumSMs * 16);
    deinterleave2_kernel<<<blocks, 256, 0, s>>>(d_in, n_frames, d_out, channel_stride);
  } else {
    const unsigned blocks = (unsigned)std::min<int64_t>(ceil_div(n_frames * n_channels, 256), kNumSMs * 16);
    deinterleave_kernel<<<blocks, 256, 0, s>>>(d_in, n_frames, n_channels, d_out, channel_stride);
  }
  SIA_CHECK_LAUNCH();
  return SIA_OK;
}

int64_t sia_num_frames(int64_t n_samples) {
  const int64_t n = n_samples < SIA_NFFT ? SIA_NFFT : n_samples;
  return (n - SIA_HOP) / SIA_HOP;
}

int64_t sia_fp_frames(const sia_fp_params *p, int64_t n_samples) {
  int rc = check_params(p);
  if (rc) return rc;
  SIA_REQUIRE(n_samples >= 0, SIA_E_INVALID, "negative track length");
  return fp_frames(p, n_samples);
}

int sia_ctx_create(int device, int64_t max_chunk_frames, sia_ctx **out) {
  SIA_REQUIRE(out != nullptr, SIA_E_INVALID, "out is NULL");
  *out = nullptr;
  int ndev = 0;
  SIA_CUDA(cudaGetDeviceCount(&ndev));
  SIA_REQUIRE(device >= 0 && device < ndev, SIA_E_INVALID, "no such CUDA device");
  SIA_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  SIA_CUDA(cudaGetDeviceProperties(&prop, device));
  SIA_REQUIRE(prop.major == 10, SIA_E_UNSUPPORTED, "sia_b200 kernels are built for sm_100a (B200) only");
  sia_ctx *c = new (std::nothrow) sia_ctx();
  SIA_REQUIRE(c != nullptr, SIA_E_NOMEM, "out of host memory");
  c->device = device;
  c->max_frames = max_chunk_frames > 0 ? max_chunk_frames : 131072;
  c->cap_peaks = c->max_frames * env_i64("SIA_PEAKS_PER_FRAME_CAP", 32);
  c->cap_chunk_hashes = c->max_frames * env_i64("SIA_HASHES_PER_FRAME_CAP", 256);
  int rc = stft_tables_create(c->tf, c->td);
  if (rc) { delete c; return rc; }
#define ALLOC(ptr, bytes)                                                      \
  do {                                                                         \
    cudaError_t _e = cudaMalloc((void **)&(ptr), (bytes));                     \
    if (_e != cudaSuccess) {                                                   \
      int _rc = cuda_fail(_e, "cudaMalloc " #ptr, __FILE__, __LINE__);         \
      sia_ctx_destroy(c);                                                      \
      return _rc;                                                              \
    }                                                                          \
  } while (0)
  ALLOC(c->spec, (size_t)c->max_frames * SIA_F_STRIDE * sizeof(float));
  ALLOC(c->bitmap, (size_t)c->max_frames * kBitmapRowWords * sizeof(uint32_t));
  ALLOC(c->row_count, (size_t)c->max_frames * sizeof(uint32_t));
  ALLOC(c->row_off, (size_t)(c->max_frames + 1) * sizeof(int64_t));
  ALLOC(c->peak_t, (size_t)c->cap_peaks * sizeof(int32_t));
  ALLOC(c->peak_f, (size_t)c->cap_peaks * sizeof(int32_t));
  ALLOC(c->pair_count, (size_t)c->cap_peaks * sizeof(uint32_t));
  ALLOC(c->pair_off, (size_t)(c->cap_peaks + 1) * sizeof(int64_t));
  ALLOC(c->scan_tmp, scan_tmp_bytes(std::max(c->cap_peaks, c->max_frames)));
  ALLOC(c->status, sizeof(int32_t));
  ALLOC(c->hash_base, sizeof(int64_t));
#undef ALLOC
  *out = c;
  return SIA_OK;
}

int sia_ctx_destroy(sia_ctx *c) {
  if (!c) return SIA_OK;
  cudaSetDevice(c->device);
  cudaDeviceSynchronize();
  stft_tables_destroy(c->tf, c->td);
  void *ptrs[] = {c->spec, c->bitmap, c->row_count, c->row_off, c->peak_t, c->peak_f, c->pair_count, c->pair_off,
                  c->scan_tmp, c->status, c->hash_base, c->d_meta, c->pcm_stage[0], c->pcm_stage[1],
                  c->hash_stage[0], c->hash_stage[1], c->t1_stage[0], c->t1_stage[1], c->digest_table};
  for (void *p : ptrs) if (p) cudaFree(p);
  if (c->h_pinned) cudaFreeHost(c->h_pinned);
  if (c->s_h2d) cudaStreamDestroy(c->s_h2d);
  if (c->s_comp) cudaStreamDestroy(c->s_comp);
  if (c->s_d2h) cudaStreamDestroy(c->s_d2h);
  collect_timing(c);
  for (cudaEvent_t e : c->ev_pool) cudaEventDestroy(e);
  delete c;
  return SIA_OK;
}

int sia_ctx_digest_table(sia_ctx *c, int enable) {
  SIA_REQUIRE(c != nullptr, SIA_E_INVALID, "ctx is NULL");
  SIA_CUDA(cudaSetDevice(c->device));
  SIA_CUDA(cudaDeviceSynchronize());
  if (!enable) {
    if (c->digest_table) cudaFree(c->digest_table);
    c->digest_table = nullptr;
    return SIA_OK;
  }
  if (c->digest_table) return SIA_OK;
  SIA_CUDA(cudaMalloc(&c->digest_table, digest_table_bytes()));
  int rc = digest_table_build(c->digest_table, nullptr);
  if (!rc && cudaDeviceSynchronize() != cudaSuccess) rc = cuda_fail(cudaGetLastError(), "digest table", __FILE__, __LINE__);
  if (rc) { cudaFree(c->digest_table); c->digest_table = nullptr; }
  return rc;
}

int sia_ctx_timing(sia_ctx *c, int enable, double *h_ms_out, int32_t *h_launches_out, int32_t n) {
  SIA_REQUIRE(c != nullptr, SIA_E_INVALID, "ctx is NULL");
  SIA_CUDA(cudaSetDevice(c->device));
  SIA_CUDA(cudaDeviceSynchronize());
  collect_timing(c);
  for (int i = 0; i < n && i < T_NCAT; ++i) {
    if (h_ms_out) h_ms_out[i] = c->ms[i];
    if (h_launches_out) h_launches_out[i] = c->launches[i];
  }
  for (int i = 0; i < T_NCAT; ++i) { c->ms[i] = 0; c->launches[i] = 0; }
  c->timing = enable != 0;
  return SIA_OK;
}

// ---- stage entry points ------------------------------------------------------------------------------

int sia_stft_db(sia_ctx *c, const int16_t *d_pcm, const int64_t *h_track_starts, const int64_t *h_track_len,
                int32_t n_tracks, const sia_fp_params *p, void *d_spec, int32_t out_type, int64_t *h_total_frames,
                void *stream) {
  SIA_REQUIRE(c && d_pcm && h_track_starts && h_track_len && d_spec, SIA_E_INVALID, "NULL argument");
  SIA_REQUIRE(n_tracks >= 0, SIA_E_INVALID, "n_tracks < 0");
  int rc = check_params(p);
  if (rc) return rc;
  SIA_CUDA(cudaSetDevice(c->device));
  cudaStream_t s = (cudaStream_t)stream;
  std::vector<int64_t> h((size_t)MetaView::size(n_tracks));
  std::vector<Chunk> one{{0, n_tracks, 0, 0, 0}};
  for (int b = 0; b < n_tracks; ++b) {
    SIA_REQUIRE(h_track_starts[b] % 8 == 0, SIA_E_INVALID, "track_starts must be multiples of 8 samples");
    SIA_REQUIRE(h_track_len[b] >= 0, SIA_E_INVALID, "negative track length");
    one[0].frames += fp_frames(p, h_track_len[b]);
  }
  fill_meta(one, p, h_track_starts, h_track_len, h.data());
  if ((rc = ensure_meta(c, h.size()))) return rc;
  SIA_CUDA(cudaMemcpyAsync(c->d_meta, h.data(), h.size() * sizeof(int64_t), cudaMemcpyHostToDevice, s));
  SIA_CUDA(cudaStreamSynchronize(s));   // h is a stack-lifetime buffer
  MetaView m(c->d_meta, n_tracks);
  if (h_total_frames) *h_total_frames = one[0].frames;
  return run_stft(c, d_pcm, m, n_tracks, one[0].frames, p, d_spec, out_type, s);
}

int sia_peaks(sia_ctx *c, const void *d_spec, int32_t in_type, const int64_t *h_track_frames, int32_t n_tracks,
              const sia_fp_params *p, int32_t *d_peak_t, int32_t *d_peak_f, int64_t cap_peaks,
              int64_t *d_track_peak_starts, int32_t *d_status, void *stream) {
  SIA_REQUIRE(c && d_spec && h_track_frames && d_peak_t && d_peak_f && d_track_peak_starts && d_status, SIA_E_INVALID,
              "NULL argument");
  int rc = check_params(p);
  if (rc) return rc;
  SIA_CUDA(cudaSetDevice(c->device));
  cudaStream_t s = (cudaStream_t)stream;
  std::vector<int64_t> h((size_t)MetaView::size(n_tracks), 0);
  MetaView hm(h.data(), n_tracks);
  int64_t fr = 0, tt = 0;
  for (int b = 0; b < n_tracks; ++b) {
    SIA_REQUIRE(h_track_frames[b] >= 1, SIA_E_INVALID, "every track has at least one frame");
    hm.frame_starts[b] = fr; hm.ttile_starts[b] = tt;
    fr += h_track_frames[b]; tt += ceil_div(h_track_frames[b], kPeakTileT);
  }
  hm.frame_starts[n_tracks] = fr; hm.ttile_starts[n_tracks] = tt;
  SIA_REQUIRE(fr <= c->max_frames, SIA_E_CAPACITY, "sia_peaks: more frames than the context workspace holds");
  if ((rc = ensure_meta(c, h.size()))) return rc;
  SIA_CUDA(cudaMemcpyAsync(c->d_meta, h.data(), h.size() * sizeof(int64_t), cudaMemcpyHostToDevice, s));
  SIA_CUDA(cudaMemsetAsync(d_status, 0, sizeof(int32_t), s));
  SIA_CUDA(cudaMemsetAsync(d_track_peak_starts, 0, sizeof(int64_t) * (n_tracks + 1), s));
  SIA_CUDA(cudaStreamSynchronize(s));
  MetaView m(c->d_meta, n_tracks);
  return run_peaks(c, d_spec, in_type, m, n_tracks, fr, tt, p, d_peak_t, d_peak_f, cap_peaks, d_track_peak_starts,
                   d_status, s);
}

int sia_pairs_sha1(sia_ctx *c, const int32_t *d_peak_t, const int32_t *d_peak_f, const int64_t *d_track_peak_starts,
                   int32_t n_tracks, int32_t fan_value, uint8_t *d_hash, int32_t *d_t1, int64_t cap_hashes,
                   int64_t *d_track_hash_starts, int32_t *d_status, void *stream) {
  SIA_REQUIRE(c && d_peak_t && d_peak_f && d_track_peak_starts && d_hash && d_t1 && d_track_hash_starts && d_status,
              SIA_E_INVALID, "NULL argument");
  SIA_REQUIRE(fan_value >= 1 && fan_value <= 64, SIA_E_INVALID, "fan_value must be in 1..64");
  SIA_CUDA(cudaSetDevice(c->device));
  cudaStream_t s = (cudaStream_t)stream;
  // the peak count lives on the device; bound the launches by the workspace capacity
  int64_t n_peaks = 0;
  SIA_CUDA(cudaMemcpyAsync(&n_peaks, d_track_peak_starts + n_tracks, sizeof(int64_t), cudaMemcpyDeviceToHost, s));
  SIA_CUDA(cudaStreamSynchronize(s));
  SIA_REQUIRE(n_peaks <= c->cap_peaks, SIA_E_CAPACITY, "sia_pairs_sha1: more peaks than the context workspace holds");
  SIA_CUDA(cudaMemsetAsync(d_status, 0, sizeof(int32_t), s));
  return run_pairs(c, d_peak_t, d_peak_f, d_track_peak_starts, n_tracks, n_peaks, fan_value, 0, nullptr, d_hash, d_t1,
                   cap_hashes, d_track_hash_starts, d_status, s);
}

// ---- whole path, device-resident PCM --------------------------------------------------------------------

int sia_fingerprint_batch(sia_ctx *c, const int16_t *d_pcm, const int64_t *h_track_starts, const int64_t *h_track_len,
                          int32_t n_tracks, const sia_fp_params *p, uint8_t *d_hash, int32_t *d_t1,
                          int64_t cap_hashes, int64_t *h_track_hash_starts, int64_t *h_total, void *stream) {
  SIA_REQUIRE(c && h_track_starts && h_track_len && h_total, SIA_E_INVALID, "NULL argument");
  SIA_REQUIRE(n_tracks >= 0, SIA_E_INVALID, "n_tracks < 0");
  SIA_REQUIRE(n_tracks == 0 || (d_pcm && d_hash && d_t1), SIA_E_INVALID, "NULL device buffer");
  int rc = check_params(p);
  if (rc) return rc;
  SIA_CUDA(cudaSetDevice(c->device));
  cudaStream_t s = (cudaStream_t)stream;
  for (int b = 0; b < n_tracks; ++b) {
    SIA_REQUIRE(h_track_starts[b] % 8 == 0, SIA_E_INVALID, "track_starts must be multiples of 8 samples");
    SIA_REQUIRE(h_track_len[b] >= 0, SIA_E_INVALID, "negative track length");
  }
  std::vector<Chunk> chunks;
  if ((rc = plan_chunks(c, p, h_track_len, n_tracks, 0, chunks))) return rc;
  size_t meta_total = 0;
  for (auto &ch : chunks) meta_total += MetaView::size(ch.b1 - ch.b0);
  if ((rc = ensure_meta(c, meta_total))) return rc;
  if ((rc = ensure_pinned(c, meta_total + 8))) return rc;
  fill_meta(chunks, p, h_track_starts, h_track_len, c->h_pinned);
  SIA_CUDA(cudaMemcpyAsync(c->d_meta, c->h_pinned, meta_total * sizeof(int64_t), cudaMemcpyHostToDevice, s));
  SIA_CUDA(cudaMemsetAsync(c->status, 0, sizeof(int32_t), s));
  SIA_CUDA(cudaMemsetAsync(c->hash_base, 0, sizeof(int64_t), s));
  for (const Chunk &ch : chunks)
    if ((rc = run_chunk(c, d_pcm, ch, p, d_hash, d_t1, cap_hashes, s))) return rc;
  // results: per-track offsets, total, status — one synchronisation
  SIA_CUDA(cudaMemcpyAsync(c->h_pinned, c->d_meta, meta_total * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
  int64_t *tail = c->h_pinned + meta_total;
  SIA_CUDA(cudaMemcpyAsync(tail, c->hash_base, sizeof(int64_t), cudaMemcpyDeviceToHost, s));
  SIA_CUDA(cudaMemcpyAsync(tail + 1, c->status, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
  SIA_CUDA(cudaStreamSynchronize(s));
  const int64_t total = tail[0];
  const int32_t status = *reinterpret_cast<int32_t *>(tail + 1);
  *h_total = total;
  if (h_track_hash_starts) {
    for (const Chunk &ch : chunks) {
      const int nb = ch.b1 - ch.b0;
      MetaView m(c->h_pinned + ch.meta_off, nb);
      for (int i = 0; i < nb; ++i) h_track_hash_starts[ch.b0 + i] = m.track_hash_starts[i];
    }
    h_track_hash_starts[n_tracks] = total;
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
  return SIA_OK;
}

// ---- whole path, host memory in and out --------------------------------------------------------------------

int sia_fingerprint_batch_host(sia_ctx *c, const int16_t *h_pcm, const int64_t *h_track_starts,
                               const int64_t *h_track_len, int32_t n_tracks, const sia_fp_params *p, uint8_t *h_hash,
                               int32_t *h_t1, int64_t cap_hashes, int64_t *h_track_hash_starts, int64_t *h_total) {
  SIA_REQUIRE(c && h_track_starts && h_track_len && h_total, SIA_E_INVALID, "NULL argument");
  SIA_REQUIRE(n_tracks >= 0, SIA_E_INVALID, "n_tracks < 0");
  SIA_REQUIRE(n_tracks == 0 || (h_pcm && h_hash && h_t1), SIA_E_INVALID, "NULL host buffer");
  int rc = check_params(p);
  if (rc) return rc;
  SIA_CUDA(cudaSetDevice(c->device));
  if (!c->s_h2d) {
    SIA_CUDA(cudaStreamCreateWithFlags(&c->s_h2d, cudaStreamNonBlocking));
    SIA_CUDA(cudaStreamCreateWithFlags(&c->s_comp, cudaStreamNonBlocking));
    SIA_CUDA(cudaStreamCreateWithFlags(&c->s_d2h, cudaStreamNonBlocking));
  }
  // The longest admissible track (max_frames frames at hop h) has (max_frames-1)*h + 4095 + h samples, 8-sample padded
  // + 8 in the staging buffer; plan_chunks keeps chunks inside.  Sized for hop 2048 at first, grown for a longer hop.
  const int64_t stage_need = (c->max_frames + 1) * (int64_t)std::max(fp_hop(p), SIA_HOP) + 3 * SIA_HOP;
  if (c->pcm_stage_samples < stage_need) {
    for (int i = 0; i < 2; ++i) {
      if (c->pcm_stage[i]) cudaFree(c->pcm_stage[i]);
      c->pcm_stage[i] = nullptr;
    }
    c->pcm_stage_samples = 0;
    for (int i = 0; i < 2; ++i) SIA_CUDA(cudaMalloc(&c->pcm_stage[i], (size_t)stage_need * sizeof(int16_t)));
    c->pcm_stage_samples = stage_need;
  }
  if (!c->hash_stage[0]) {
    for (int i = 0; i < 2; ++i) {
      SIA_CUDA(cudaMalloc(&c->hash_stage[i], (size_t)c->cap_chunk_hashes * SIA_HASH_BYTES));
      SIA_CUDA(cudaMalloc(&c->t1_stage[i], (size_t)c->cap_chunk_hashes * sizeof(int32_t)));
    }
  }
  for (int b = 0; b < n_tracks; ++b) SIA_REQUIRE(h_track_len[b] >= 0, SIA_E_INVALID, "negative track length");

  std::vector<Chunk> chunks;
  if ((rc = plan_chunks(c, p, h_track_len, n_tracks, c->pcm_stage_samples, chunks))) return rc;
  const int nchunks = (int)chunks.size();
  size_t meta_total = 0;
  for (auto &ch : chunks) meta_total += MetaView::size(ch.b1 - ch.b0);
  // device sample offset of every track inside its chunk's staging buffer; tracks that are contiguous
  // (and equally aligned) on the host stay contiguous so that one copy moves the run
  std::vector<int64_t> dev_start(n_tracks);
  struct Copy { int64_t h_off, d_off, n; };
  std::vector<std::vector<Copy>> copies(nchunks);
  for (int ci = 0; ci < nchunks; ++ci) {
    const Chunk &ch = chunks[ci];
    int64_t d = 0;
    for (int b = ch.b0; b < ch.b1; ++b) {
      bool merged = false;
      if (!copies[ci].empty()) {
        Copy &last = copies[ci].back();
        const int64_t gap = h_track_starts[b] - (last.h_off + last.n);
        const int64_t d_here = last.d_off + last.n + gap;
        if (gap >= 0 && gap <= 8 && d_here % 8 == 0) {
          last.n += gap + h_track_len[b];
          dev_start[b] = d_here;
          d = last.d_off + last.n;
          merged = true;
        }
      }
      if (!merged) {
        d = (d + 7) / 8 * 8;
        dev_start[b] = d;
        copies[ci].push_back({h_track_starts[b], d, h_track_len[b]});
        d += h_track_len[b];
      }
    }
    SIA_REQUIRE(d <= c->pcm_stage_samples, SIA_E_CAPACITY, "chunk PCM exceeds the staging buffer");
  }
  if ((rc = ensure_meta(c, meta_total))) return rc;
  if ((rc = ensure_pinned(c, 2 * meta_total + 2 * (size_t)nchunks + 8))) return rc;
  int64_t *h_meta_in = c->h_pinned;                 // upload image
  int64_t *h_meta_out = c->h_pinned + meta_total;   // per-chunk readback of track_hash_starts etc.
  int64_t *h_counts = h_meta_out + meta_total;      // [nchunks] hashes per chunk
  int32_t *h_status = reinterpret_cast<int32_t *>(h_counts + nchunks);
  fill_meta(chunks, p, dev_start.data(), h_track_len, h_meta_in);
  SIA_CUDA(cudaMemcpyAsync(c->d_meta, h_meta_in, meta_total * sizeof(int64_t), cudaMemcpyHostToDevice, c->s_comp));
  SIA_CUDA(cudaMemsetAsync(c->status, 0, sizeof(int32_t), c->s_comp));

  // Every exit below goes through ONE epilogue that waits for the three streams (async copies into the caller's host
  // buffers must not outlive the call, whatever failed) and destroys the events.
  std::vector<cudaEvent_t> ev_h2d(nchunks, nullptr), ev_comp(nchunks, nullptr), ev_d2h(nchunks, nullptr);
  auto epilogue = [&](int code) {
    cudaStreamSynchronize(c->s_comp); cudaStreamSynchronize(c->s_d2h); cudaStreamSynchronize(c->s_h2d);
    for (int i = 0; i < nchunks; ++i)
      for (cudaEvent_t e : {ev_h2d[i], ev_comp[i], ev_d2h[i]}) if (e) cudaEventDestroy(e);
    return code;
  };

  int64_t out_base = 0;   // rows already placed in h_hash
  bool overflow = false;
  auto drain = [&](int ci) -> int {   // issue the D2H of chunk ci once its count is known
    SIA_CUDA(cudaEventSynchronize(ev_comp[ci]));
    const int64_t n = h_counts[ci];
    const Chunk &ch = chunks[ci];
    const int nb = ch.b1 - ch.b0;
    MetaView m(h_meta_out + ch.meta_off, nb);
    if (h_track_hash_starts)
      for (int i = 0; i < nb; ++i) h_track_hash_starts[ch.b0 + i] = out_base + m.track_hash_starts[i];
    if (n > c->cap_chunk_hashes || out_base + n > cap_hashes) overflow = true;
    if (!overflow && n > 0) {
      SIA_CUDA(cudaMemcpyAsync(h_hash + out_base * SIA_HASH_BYTES, c->hash_stage[ci & 1], (size_t)n * SIA_HASH_BYTES,
                               cudaMemcpyDeviceToHost, c->s_d2h));
      SIA_CUDA(cudaMemcpyAsync(h_t1 + out_base, c->t1_stage[ci & 1], (size_t)n * sizeof(int32_t),
                               cudaMemcpyDeviceToHost, c->s_d2h));
    }
    SIA_CUDA(cudaEventRecord(ev_d2h[ci], c->s_d2h));
    out_base += n;
    return SIA_OK;
  };

  auto pipeline = [&]() -> int {
  auto mkev = [&](cudaEvent_t &e) { return cudaEventCreateWithFlags(&e, cudaEventDisableTiming); };
  for (int i = 0; i < nchunks; ++i) { SIA_CUDA(mkev(ev_h2d[i])); SIA_CUDA(mkev(ev_comp[i])); SIA_CUDA(mkev(ev_d2h[i])); }
  for (int ci = 0; ci < nchunks; ++ci) {
    const Chunk &ch = chunks[ci];
    const int nb = ch.b1 - ch.b0;
    // H2D of chunk ci into staging[ci&1]: the kernels of chunk ci-2 must be done with it
    if (ci >= 2) SIA_CUDA(cudaStreamWaitEvent(c->s_h2d, ev_comp[ci - 2], 0));
    for (const Copy &cp : copies[ci])
      SIA_CUDA(cudaMemcpyAsync(c->pcm_stage[ci & 1] + cp.d_off, h_pcm + cp.h_off, (size_t)cp.n * sizeof(int16_t),
                               cudaMemcpyHostToDevice, c->s_h2d));
    SIA_CUDA(cudaEventRecord(ev_h2d[ci], c->s_h2d));
    // kernels of chunk ci: need its PCM, and the output staging[ci&1] drained (D2H of chunk ci-2)
    SIA_CUDA(cudaStreamWaitEvent(c->s_comp, ev_h2d[ci], 0));
    if (ci >= 2) {
      if ((rc = drain(ci - 2))) return rc;
      SIA_CUDA(cudaStreamWaitEvent(c->s_comp, ev_d2h[ci - 2], 0));
    }
    SIA_CUDA(cudaMemsetAsync(c->hash_base, 0, sizeof(int64_t), c->s_comp));
    if ((rc = run_chunk(c, c->pcm_stage[ci & 1], ch, p, c->hash_stage[ci & 1], c->t1_stage[ci & 1],
                        c->cap_chunk_hashes, c->s_comp))) return rc;
    MetaView dm(c->d_meta + ch.meta_off, nb);
    MetaView hm(h_meta_out + ch.meta_off, nb);
    SIA_CUDA(cudaMemcpyAsync(hm.track_hash_starts, dm.track_hash_starts, sizeof(int64_t) * (nb + 1),
                             cudaMemcpyDeviceToHost, c->s_comp));
    SIA_CUDA(cudaMemcpyAsync(h_counts + ci, c->hash_base, sizeof(int64_t), cudaMemcpyDeviceToHost, c->s_comp));
    SIA_CUDA(cudaEventRecord(ev_comp[ci], c->s_comp));
  }
  for (int ci = std::max(0, nchunks - 2); ci < nchunks; ++ci)
    if ((rc = drain(ci))) return rc;
  SIA_CUDA(cudaMemcpyAsync(h_status, c->status, sizeof(int32_t), cudaMemcpyDeviceToHost, c->s_comp));
  SIA_CUDA(cudaStreamSynchronize(c->s_comp));
  SIA_CUDA(cudaStreamSynchronize(c->s_d2h));
  SIA_CUDA(cudaStreamSynchronize(c->s_h2d));
  return SIA_OK;
  };
  if ((rc = epilogue(pipeline()))) return rc;
  *h_total = out_base;
  if (h_track_hash_starts) h_track_hash_starts[n_tracks] = out_base;
  if (*h_status & 1) {
    set_error("peak workspace overflow: more than SIA_PEAKS_PER_FRAME_CAP (default 32) peaks per frame on average");
    return SIA_E_CAPACITY;
  }
  if ((*h_status & 2) || overflow) {
    set_error("hash output capacity exceeded (cap_hashes, or SIA_HASHES_PER_FRAME_CAP per chunk); *h_total holds the "
              "required number of rows");
    return SIA_E_CAPACITY;
  }
  return SIA_OK;
}

}  // extern "C"
