// Internal launch interfaces of the fingerprint kernels (K1-K3).
#pragma once
#include "sia_common.cuh"

namespace sia {

template <typename T>
struct StftTables {
  void *base = nullptr;
  const void *win2 = nullptr;  // [2048] (w[2n], w[2n+1])
  const void *twA = nullptr;   // [16][128] W2048^(t*ka)
  const void *twB = nullptr;   // [16][8]   W128^(c*kb)
  const void *twP = nullptr;   // [1025]    W4096^k
};

struct StftLaunch {
  const int16_t *d_pcm;
  const int64_t *d_track_starts;  // [n_tracks]   samples
  const int64_t *d_track_len;     // [n_tracks]   samples
  const int64_t *d_frame_starts;  // [n_tracks+1] rows
  int n_tracks;
  int64_t total_frames;
  int frames_per_cta;
  void *d_spec;
  int out_type;   // SIA_F32 / SIA_F64
  int compute;    // SIA_F32 / SIA_F64
  double Fs;
  int hop;        // frame k of a track starts at sample k * hop, 1..4096 (SIA_HOP: the half-block staging)
};

int stft_tables_create(StftTables<float> &f, StftTables<double> &d);
void stft_tables_destroy(StftTables<float> &f, StftTables<double> &d);
int stft_db_launch(const StftLaunch &a, const StftTables<float> &tf, const StftTables<double> &td, cudaStream_t s);
double hann_power_sum();

// ---- K2 ------------------------------------------------------------------------------------
struct PeaksLaunch {
  const void *d_spec;
  int in_type;                    // SIA_F32 / SIA_F64
  const int64_t *d_frame_starts;  // [n_tracks+1]
  const int64_t *d_ttile_starts;  // [n_tracks+1] prefix of per-track time-tile counts
  int n_tracks;
  int64_t total_frames;
  int64_t total_ttiles;
  double amp_min;
  int connectivity;               // 1 diamond, 2 square
  int nbhd;
  uint32_t *d_bitmap;             // [total_frames][kBitmapRowWords]
};
constexpr int kBitmapRowWords = 88;   // row stride of the peak bitmap: 22 strips x 4 words (striped) >= 65 (plain)
constexpr int kPeakTileT = 64;    // output rows per tile
constexpr int kPeakTileF = 128;   // output bins per tile
// *striped tells which bitmap layout was written (see peaks.cu)
int peaks_bitmap_launch(const PeaksLaunch &a, cudaStream_t s, bool *striped);

// Streaming (stream.cu): of segment b (rows [frame_starts[b], frame_starts[b+1])) only the segment-local rows
// [emit_lo[b], emit_hi[b]) yield peaks, their t is t_base[b] + local row, and they are placed peak_off[b] entries after
// their scan offset.  The caller then fills the segments' peak starts itself (track_peak_starts may be NULL).
struct PeakWindow {
  const int64_t *frame_starts;   // [n+1]
  const int64_t *emit_lo, *emit_hi, *t_base, *peak_off;   // [n]
  int n;
};

// bitmap -> ordered (t, f) lists.  d_row_count/d_row_off: [total_frames(+1)] workspaces.
int peaks_rowcount_launch(const uint32_t *d_bitmap, bool striped, int64_t total_frames, uint32_t *d_row_count,
                          cudaStream_t s, const PeakWindow *win = nullptr);
int peaks_extract_launch(const uint32_t *d_bitmap, bool striped, const int64_t *d_row_off,
                         const int64_t *d_frame_starts, int n_tracks, int64_t total_frames, int64_t peak_base, int32_t *d_peak_t,
                         int32_t *d_peak_f, int64_t cap_peaks, int64_t *d_track_peak_starts, int32_t *d_status,
                         cudaStream_t s, const PeakWindow *win = nullptr);

// ---- K3 ------------------------------------------------------------------------------------
// d_n_peaks: device scalar (total peaks, = track_peak_starts[n_tracks]); launches are sized by n_peaks_max.
// d_final_t (streaming, [n_tracks]): anchors of track b with t > d_final_t[b] and fewer than fan_value-1 peaks behind
// them in the track are not final yet and get no pairs; NULL = every anchor is final.
int pairs_count_launch(const int32_t *d_peak_t, const int64_t *d_track_peak_starts, int n_tracks,
                       int64_t n_peaks_max, int fan_value, uint32_t *d_pair_count, cudaStream_t s,
                       const int64_t *d_final_t = nullptr);
int pairs_sha1_launch(const int32_t *d_peak_t, const int32_t *d_peak_f, const int64_t *d_track_peak_starts,
                      int n_tracks, int64_t n_peaks_max, int fan_value, const uint32_t *d_pair_count,
                      const int64_t *d_pair_off, int64_t hash_base_static, const int64_t *d_hash_base,
                      const void *d_digest_table, uint8_t *d_hash, int32_t *d_t1, int64_t cap_hashes,
                      int64_t *d_track_hash_starts, int32_t *d_status, cudaStream_t s);
// optional digest table of the whole pre-image space (pairs_sha1.cu): NULL = compute every digest
size_t digest_table_bytes();
int digest_table_build(void *d_table, cudaStream_t s);

}  // namespace sia
