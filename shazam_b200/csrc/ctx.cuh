// The fingerprinting context (sia_ctx) shared by the batch path (api.cu) and the streaming path (stream.cu):
// chunk workspaces, pinned scratch, per-kernel timers.
#pragma once
#include "sia_common.cuh"
#include "stft.cuh"

#include <vector>

// timer categories of sia_ctx_timing
enum { T_STFT = 0, T_PEAKS = 1, T_COMPACT = 2, T_PAIRS = 3, T_SCAN = 4, T_STREAM = 5, T_NCAT = 6 };

struct TimedSpan { cudaEvent_t a, b; int cat; };

struct sia_ctx {
  int device = 0;
  int64_t max_frames = 0;
  int64_t cap_peaks = 0;
  int64_t cap_chunk_hashes = 0;
  sia::StftTables<float> tf;
  sia::StftTables<double> td;
  // chunk workspace
  float *spec = nullptr;
  uint32_t *bitmap = nullptr;
  uint32_t *row_count = nullptr;
  int64_t *row_off = nullptr;
  int32_t *peak_t = nullptr, *peak_f = nullptr;
  uint32_t *pair_count = nullptr;
  int64_t *pair_off = nullptr;
  void *scan_tmp = nullptr;
  int32_t *status = nullptr;      // device flag word
  int64_t *hash_base = nullptr;   // device scalar: running output offset
  void *digest_table = nullptr;   // optional: sha1 of every (f1, f2, dt) the pipeline can produce (sia_ctx_digest_table)
  // batch metadata (grown on demand)
  int64_t *d_meta = nullptr;
  size_t d_meta_cap = 0;
  // host pipeline
  cudaStream_t s_h2d = nullptr, s_comp = nullptr, s_d2h = nullptr;
  int16_t *pcm_stage[2] = {nullptr, nullptr};
  int64_t pcm_stage_samples = 0;
  uint8_t *hash_stage[2] = {nullptr, nullptr};
  int32_t *t1_stage[2] = {nullptr, nullptr};
  int64_t *h_pinned = nullptr;    // pinned scratch: counts and track_hash_starts per chunk
  size_t h_pinned_cap = 0;
  // timing
  bool timing = false;
  std::vector<TimedSpan> spans;
  std::vector<cudaEvent_t> ev_pool;
  double ms[T_NCAT] = {};
  int launches[T_NCAT] = {};
};

namespace sia {

// CUDA events around the launches of one category on stream s (recorded only while timing is enabled)
struct Timer {
  sia_ctx *c; cudaStream_t s; int cat; int nlaunch; cudaEvent_t a = nullptr, b = nullptr;
  Timer(sia_ctx *c_, cudaStream_t s_, int cat_, int nlaunch_) : c(c_), s(s_), cat(cat_), nlaunch(nlaunch_) {
    c->launches[cat] += nlaunch;
    if (!c->timing) return;
    auto get = [&]() {
      cudaEvent_t e;
      if (!c->ev_pool.empty()) { e = c->ev_pool.back(); c->ev_pool.pop_back(); } else cudaEventCreate(&e);
      return e;
    };
    a = get(); b = get();
    cudaEventRecord(a, s);
  }
  ~Timer() {
    if (!c->timing) return;
    cudaEventRecord(b, s);
    c->spans.push_back({a, b, cat});
  }
};

int check_params(const sia_fp_params *p);
// Frame geometry of parameters that passed check_params: noverlap = int(wsize * wratio) (truncated, like Python's
// int()), frame k of a track starts at sample k * hop, and a track of n samples has 1 + (max(n, 4096) - 4096) / hop
// frames (mlab.specgram: a short input is zero-padded to one frame, a trailing partial frame is dropped).
inline int fp_hop(const sia_fp_params *p) { return SIA_NFFT - (int32_t)(SIA_NFFT * p->wratio); }
inline int64_t fp_frames(const sia_fp_params *p, int64_t n_samples) {
  return 1 + ((n_samples < SIA_NFFT ? SIA_NFFT : n_samples) - SIA_NFFT) / fp_hop(p);
}
int ensure_meta(sia_ctx *c, size_t n_i64);     // d_meta holds at least n_i64 int64
int ensure_pinned(sia_ctx *c, size_t n_i64);   // h_pinned holds at least n_i64 int64

}  // namespace sia
