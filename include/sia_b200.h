/* sia_b200.h — C ABI of the B200-native SIA fingerprint-and-match path.
 *
 * The reference (CarlosArturoMe/shazam) is pure Python and has no FFI; its
 * plug-in surface is the module-level functions `fingerprint`, `get_2D_peaks`,
 * `generate_hashes` (__init__.py:116-245), `return_matches`, `align_matches`
 * (recognizer.py:222-338) and the duck-typed database backend
 * (mysql_database.py:28-255) selected through `DATABASES`/`get_database`
 * (__init__.py:24-27,54-67).  This header is what a ctypes stub behind those
 * names binds (see INTEGRATION.md); each entry point cites the reference
 * code it replaces.
 *
 * Conventions
 *  - plain pointers and sizes only; no C++/torch types cross the boundary;
 *  - every function returns 0 on success, <0 on error (SIA_E_*), never throws;
 *    sia_last_error() returns a thread-local message for the last failure;
 *  - `d_` parameters are DEVICE pointers (cudaMalloc / torch CUDA tensors),
 *    `h_` parameters are HOST pointers (pinned for best throughput);
 *  - the caller owns all I/O buffers; the library owns workspaces and index
 *    storage behind opaque handles; one context per device; calls on one
 *    handle must be serialised by the caller;
 *  - `stream` is a cudaStream_t passed as void* (NULL = the legacy default
 *    stream).  Device-pointer entry points are stream-ordered and do not
 *    synchronise unless stated.
 *
 * Data formats
 *  - PCM: int16 mono, tracks concatenated; track b occupies samples
 *    [track_starts[b], track_starts[b] + track_len[b]).  track_starts[b] must be
 *    a multiple of 8 samples (16-byte aligned loads); gaps are never read.
 *  - spectrogram: TIME-major, row g = frame (track-concatenated), SIA_F_STRIDE
 *    values per row, bins 0..2048 valid (the transpose of the reference's
 *    [freq][time] array, __init__.py:232-241).
 *  - hash: the first 10 bytes of sha1("f1|f2|dt") — BINARY(10) in
 *    mysql_database.py:49; hex(hash) is the reference's 20-char string.
 */
#ifndef SIA_B200_H
#define SIA_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SIA_NFFT        4096   /* DEFAULT_WINDOW_SIZE, __init__.py:43 */
#define SIA_HOP         2048   /* NFFT * DEFAULT_OVERLAP_RATIO(0.5), __init__.py:44 */
#define SIA_NBINS       2049
#define SIA_F_STRIDE    2080   /* row stride (values) of device spectrograms: 65*32 */
#define SIA_ROW_WORDS   65     /* 32-bit words per row of the peak bitmap */
#define SIA_HASH_BYTES  10     /* FINGERPRINT_REDUCTION(20 hex chars)/2, __init__.py:51 */
#define SIA_MAX_DT      200    /* MAX_HASH_TIME_DELTA, __init__.py:50 */
#define SIA_MAX_NBHD    64     /* largest PEAK_NEIGHBORHOOD_SIZE supported (reference: 10); 64 frames are ~3 s at
                                 * hop 2048, against MAX_HASH_TIME_DELTA = 200 frames */

enum {
  SIA_OK = 0,
  SIA_E_INVALID = -1,     /* bad argument */
  SIA_E_CUDA = -2,        /* CUDA runtime error (message has the detail) */
  SIA_E_CAPACITY = -3,    /* an output or workspace capacity was exceeded; see message */
  SIA_E_NOMEM = -4,
  SIA_E_UNSUPPORTED = -5  /* parameter combination outside the CUDA path (e.g. wsize != 4096) */
};

enum { SIA_F32 = 0, SIA_F64 = 1 };  /* arithmetic / storage type selectors */

typedef struct sia_ctx sia_ctx;       /* per-device fingerprinting context */
typedef struct sia_index sia_index;   /* per-device fingerprint index shard */

const char *sia_last_error(void);
int sia_version(void);

/* ---- parameters of fingerprint(), __init__.py:212-217 and constants :40-51 -------- */
typedef struct sia_fp_params {
  double  Fs;            /* sampling rate; enters only as the 1/Fs PSD scale */
  int32_t wsize;         /* must be 4096 */
  double  wratio;        /* DEFAULT_OVERLAP_RATIO 0.5: noverlap = (int32_t)(4096.0 * wratio) (Python's
                          * int(wsize * wratio)) must be 0..4095; frame k of a track starts at sample k * hop,
                          * hop = 4096 - noverlap.  noverlap >= 4096 or NaN: SIA_E_INVALID; noverlap < 0:
                          * SIA_E_UNSUPPORTED.  Peak times, t1 and dt <= MAX_HASH_TIME_DELTA count frames of this hop:
                          * an index is built and queried at one wratio.  Offsets stored in an index are < 2^24, so
                          * a track inserted there has at most 2^24 frames (2^24 * hop samples; ~380 s at hop 1). */
  int32_t fan_value;     /* DEFAULT_FAN_VALUE 5; partners per peak = fan_value-1; <= 64 */
  double  amp_min;       /* DEFAULT_AMP_MIN 10 (dB); negative values enable the erosion term */
  int32_t connectivity;  /* CONNECTIVITY_MASK: 2 = square (reference default), 1 = diamond */
  int32_t nbhd;          /* PEAK_NEIGHBORHOOD_SIZE 10; 1..SIA_MAX_NBHD (64) with either connectivity: the window
                          * (2*nbhd+1 square, or |dt| + |df| <= nbhd) is clipped to the track's frames and bins
                          * 0..2048; nbhd < 1 or > 64: SIA_E_INVALID */
  int32_t compute;       /* SIA_F64 (default; |dB error| << 1e-3 on every bin) or SIA_F32 */
} sia_fp_params;

void sia_fp_params_default(sia_fp_params *p);

/* ---- context ------------------------------------------------------------------------- */
/* max_chunk_frames: spectrogram rows the workspace holds at once (0 = default 131072);
 * the longest single track must fit.  Allocates ~ max_chunk_frames * 8.6 KB. */
int sia_ctx_create(int device, int64_t max_chunk_frames, sia_ctx **out);
int sia_ctx_destroy(sia_ctx *ctx);

/* K3 as a gather: build (enable != 0) or free the per-context table of sha1("f1|f2|dt")[:10] for EVERY message the
 * pipeline can produce (f1, f2 in 0..2048, dt in 0..200: 8.4e8 entries of 16 bytes = 13.5 GB, filled once by the SHA-1
 * kernel in ~50 ms).  With the table generate_hashes (__init__.py:198-208) costs one DRAM sector per hash instead of 80
 * SHA-1 rounds; results are identical (the table IS the kernel's output).  Synchronous. */
int sia_ctx_digest_table(sia_ctx *ctx, int enable);

/* frames mlab.specgram yields for a track of n samples (short input -> 1 padded frame) */
int64_t sia_num_frames(int64_t n_samples);
/* the same at the hop of p: 1 + (max(n, 4096) - 4096) / hop; <0 (SIA_E_*, sia_last_error) if p is rejected or
 * n_samples < 0.  Host only: needs no device. */
int64_t sia_fp_frames(const sia_fp_params *p, int64_t n_samples);

/* De-interleave decoded PCM on the device — the `data[chn::n_channels]` of read(), __init__.py:91-95:
 * d_out[c * channel_stride + i] = d_in[i * n_channels + c] for i < n_frames, c < n_channels.  channel_stride >=
 * n_frames (a multiple of 8 keeps every channel 16-byte aligned for K1).  Stream-ordered. */
int sia_deinterleave_i16(const int16_t *d_in, int64_t n_frames, int32_t n_channels, int16_t *d_out,
                         int64_t channel_stride, void *stream);

/* ---- stage entry points (parity tests drive these one by one) -------------------------- */

/* K1. Replaces mlab.specgram(...)[0] + the dB transform, __init__.py:232-241.
 * d_spec receives total_frames rows of SIA_F_STRIDE values (float if out_type==SIA_F32,
 * double if SIA_F64).  h_track_starts/h_track_len: host arrays, n_tracks entries. */
int sia_stft_db(sia_ctx *ctx, const int16_t *d_pcm, const int64_t *h_track_starts,
                const int64_t *h_track_len, int32_t n_tracks, const sia_fp_params *p,
                void *d_spec, int32_t out_type, int64_t *h_total_frames, void *stream);

/* K2. Replaces get_2D_peaks, __init__.py:116-177.  d_spec as produced by K1 (in_type
 * says float/double).  Peaks are written per track in (t asc, f asc) order — the order
 * generate_hashes establishes with its stable sort (__init__.py:194-195).
 * d_peak_t: frame index within the track; d_peak_f: bin.  d_track_peak_starts: n_tracks+1
 * prefix offsets into the peak arrays.  Counts stay on the device; when the number of
 * peaks exceeds cap_peaks the excess is dropped and d_status[0] is set to 1. */
int sia_peaks(sia_ctx *ctx, const void *d_spec, int32_t in_type, const int64_t *h_track_frames,
              int32_t n_tracks, const sia_fp_params *p, int32_t *d_peak_t, int32_t *d_peak_f,
              int64_t cap_peaks, int64_t *d_track_peak_starts, int32_t *d_status, void *stream);

/* K3. Replaces generate_hashes, __init__.py:179-210, on peaks already in (t, f) order.
 * Output order is the reference's list order (i major, j minor).  d_hash: [cap][10] bytes,
 * d_t1: [cap].  d_track_hash_starts: n_tracks+1 prefix offsets.  d_status[0] flags: 2 = output overflow, 4 = a peak
 * bin outside 0..99999 (the message would not fit one SHA-1 block the way the kernel packs it; such rows are skipped
 * and the caller must treat the call as failed). */
int sia_pairs_sha1(sia_ctx *ctx, const int32_t *d_peak_t, const int32_t *d_peak_f,
                   const int64_t *d_track_peak_starts, int32_t n_tracks, int32_t fan_value,
                   uint8_t *d_hash, int32_t *d_t1, int64_t cap_hashes,
                   int64_t *d_track_hash_starts, int32_t *d_status, void *stream);

/* ---- whole path ----------------------------------------------------------------------- */

/* Replaces the per-channel body of fingerprint() (__init__.py:212-245) for a batch of
 * tracks — the unit _fingerprint_worker/imap_unordered distributes (__init__.py:271,357).
 * PCM resident on the device.  Tracks are processed in chunks of <= max_chunk_frames.
 * Outputs on the device; h_track_hash_starts (n_tracks+1, host) and *h_total are filled
 * after one synchronisation at the end.  Returns SIA_E_CAPACITY if cap_hashes was too
 * small (h_total then holds the required size). */
int sia_fingerprint_batch(sia_ctx *ctx, const int16_t *d_pcm, const int64_t *h_track_starts,
                          const int64_t *h_track_len, int32_t n_tracks, const sia_fp_params *p,
                          uint8_t *d_hash, int32_t *d_t1, int64_t cap_hashes,
                          int64_t *h_track_hash_starts, int64_t *h_total, void *stream);

/* Same, end to end from HOST memory: pinned (or pageable) PCM in, digests out to host
 * memory, H2D / kernels / D2H pipelined over internal streams.  Synchronous. */
int sia_fingerprint_batch_host(sia_ctx *ctx, const int16_t *h_pcm, const int64_t *h_track_starts,
                               const int64_t *h_track_len, int32_t n_tracks, const sia_fp_params *p,
                               uint8_t *h_hash, int32_t *h_t1, int64_t cap_hashes,
                               int64_t *h_track_hash_starts, int64_t *h_total);

/* per-kernel device time (ms, CUDA events on the launching stream) accumulated since the
 * last reset; order: stft, peaks(bitmap), peaks(compact), pairs+sha1, scans, stream-state copies
 * (staging, row assembly, peak splice and commit of sia_stream_push).  n <= 8. */
int sia_ctx_timing(sia_ctx *ctx, int enable, double *h_ms_out, int32_t *h_launches_out, int32_t n);

/* ---- streaming: many concurrent streams, fed block by block ------------------------------------------------------
 * A stream handle holds n_streams independent streams on one context.  Each push gives every stream a block of int16
 * PCM (possibly empty); h_end[b] != 0 marks the block as stream b's last, after which the stream starts over at frame 0.
 * A push returns, per stream, the hashes that became final in it: with F complete frames so far, rows up to
 * H = F - 1 - nbhd have their whole neighbourhood, their peaks are final, and an anchor is final once it has
 * fan_value - 1 peaks behind it or t <= H - MAX_HASH_TIME_DELTA; at the end everything is.  So for ANY cut of a
 * stream's PCM into blocks, the concatenation of everything emitted up to and including the end push equals
 * sia_fingerprint_batch on the whole PCM with the same parameters (digests, t1 = frame index from the stream's start,
 * order), short-input padding included.  Streams longer than the context workspace are fine: a push only needs the
 * carried 2*nbhd rows + its new frames of each stream to fit max_chunk_frames.
 *
 * The handle keeps per-stream state in HBM (allocated at create, two copies: ~2 * (8 KB + nbhd * 16.6 KB) per stream,
 * 2.1 MB at nbhd 64, plus one max_chunk_frames spectrogram for new rows) and uses its context's workspaces: calls on a context and its
 * stream handles must be serialised by the caller, and stream handles are destroyed before their context.
 * Parameters as sia_fingerprint_batch (wsize 4096 only). */
typedef struct sia_stream sia_stream;
int sia_stream_create(sia_ctx *ctx, int32_t n_streams, const sia_fp_params *p, sia_stream **out);
int sia_stream_destroy(sia_stream *st);
/* Block b of the push: samples [h_block_starts[b], +h_block_len[b]) of d_pcm (starts multiples of 8, as in the batch
 * path; ignored for empty blocks).  h_end: n_streams flags, or NULL for none.  Outputs like sia_fingerprint_batch:
 * digests and t1 on the device, h_stream_hash_starts (n_streams+1, optional) and *h_total on the host after ONE
 * synchronisation.  A push that fails leaves every stream exactly as it was: SIA_E_CAPACITY when cap_hashes is too
 * small (*h_total = rows needed), when a stream's carried + new rows exceed the workspace (push smaller blocks) or the
 * peak workspace overflows; the push can then be retried. */
int sia_stream_push(sia_stream *st, const int16_t *d_pcm, const int64_t *h_block_starts, const int64_t *h_block_len,
                    const uint8_t *h_end, uint8_t *d_hash, int32_t *d_t1, int64_t cap_hashes,
                    int64_t *h_stream_hash_starts, int64_t *h_total, void *stream);

/* ---- noise-robustness harness (SURVEY §8f-3) -------------------------------------------------------------------- */
/* get_noise_from_sound + the mix (recognizer_test.py:426-435, 554) for a batch of clips: clip c reads n_samples int16
 * at d_signal + c * signal_stride and n_samples float noise samples at d_noise + c * noise_stride, and writes
 * round(signal + noise * RMS_n / RMS_noise), RMS_n = RMS_signal / 10^(SNR/20), saturated to int16, at d_out + c *
 * out_stride (a multiple of 8 keeps the clips aligned for K1).  d_scale_out (optional, n_clips doubles): the factor
 * applied to each clip's noise.  Stream-ordered. */
int sia_mix_noise(int device, const int16_t *d_signal, int64_t signal_stride, const float *d_noise, int64_t noise_stride,
                  int32_t n_clips, int64_t n_samples, double snr_db, int16_t *d_out, int64_t out_stride,
                  double *d_scale_out, void *stream);

/* ---- index (replaces the fingerprints table + SELECT_MULTIPLE + align_matches) --------- */

/* One shard of the `fingerprints` table (mysql_database.py:46-59): rows
 * (hash BINARY(10), song_id MEDIUMINT UNSIGNED (< 2^24), offset INT UNSIGNED (< 2^24 here)),
 * UNIQUE(song_id, offset, hash) -> set semantics (INSERT IGNORE, :62-68).
 * Storage: every distinct hash once (16-byte key entry: hash + start of its posting run) and one packed 8-byte
 * posting (song_id, offset) per row — 8 bytes per row + 16 per distinct hash, so the 100 000-track index of
 * BASELINE.json configs[3] (8e9 rows) is 64 GB of postings and fits one B200.  capacity_rows postings are
 * allocated up front; key table, directory and pending buffers grow on demand. */
int sia_index_create(int device, int64_t capacity_rows, sia_index **out);
int sia_index_destroy(sia_index *ix);

/* insert_hashes(song_id, hashes), mysql_database.py:167-181.  Rows are appended to a
 * pending run; they become visible to queries after sia_index_finalize.  Stream-ordered on
 * `stream` (any stream: finalize waits for the last insert). */
int sia_index_insert(sia_index *ix, int32_t song_id, const uint8_t *d_hash, const int32_t *d_off,
                     int64_t n, void *stream);
/* rows for many songs at once: d_song[n] gives each row's song id */
int sia_index_insert_rows(sia_index *ix, const int32_t *d_song, const uint8_t *d_hash,
                          const int32_t *d_off, int64_t n, void *stream);
int sia_index_insert_host(sia_index *ix, int32_t song_id, const uint8_t *h_hash, const int32_t *h_off,
                          int64_t n);

/* Merge the pending rows into the table: sorts ONLY the pending rows, drops duplicates (of each other and of stored
 * rows), and shifts the stored postings in place — the cost is O(pending log) + one pass over the part of the table
 * behind the first inserted row, with scratch proportional to the pending rows (the reference commits per song,
 * __init__.py:381-386).  *h_rows = rows now stored.  Synchronous; runs on the legacy default stream. */
int sia_index_finalize(sia_index *ix, int64_t *h_rows);
int64_t sia_index_rows(const sia_index *ix);
int64_t sia_index_keys(const sia_index *ix);       /* distinct hashes stored */
int32_t sia_index_max_song(const sia_index *ix);   /* largest song id inserted so far (as of the last finalize) */

/* Give back everything that is not the table itself: pending buffers, the second key buffer, build / lookup / vote
 * scratch (all of it is re-allocated on demand by the next insert, finalize or query).  Synchronous. */
int sia_index_trim(sia_index *ix);

/* DELETE FROM songs WHERE ... with ON DELETE CASCADE on fingerprints (mysql_database.py:56-57,
 * 132-139): remove every stored row of the listed songs.  *h_rows = rows left.  Synchronous. */
int sia_index_delete_songs(sia_index *ix, const int32_t *h_song_ids, int32_t n, int64_t *h_rows);

/* Rows [first_row, first_row+n) of the sorted table back in the schema's vocabulary (hash BINARY(10),
 * song_id, offset) — for dumping the index to / seeding it from the MySQL `fingerprints` table
 * (mysql_database.py:46-59).  Stream-ordered; rows come in (hash, song_id, offset) order. */
int sia_index_export(sia_index *ix, int64_t first_row, int64_t n, uint8_t *d_hash, int32_t *d_song, int32_t *d_off,
                     void *stream);

/* SELECT HEX(hash), song_id, offset WHERE hash IN (...) (recognizer.py:60-64, 252-259):
 * every stored row whose hash is in the list of n DISTINCT hashes.  Row order: by hash
 * (h_row_hashidx gives the position of the row's hash in h_hash), then (song_id, offset); the host
 * layer re-orders to IN-list order.  Fills up to cap rows; *h_nrows = total. */
int sia_index_select_host(sia_index *ix, const uint8_t *h_hash, int64_t n, int32_t *h_row_hashidx,
                          int32_t *h_row_song, int32_t *h_row_off, int64_t cap, int64_t *h_nrows);

/* return_matches + the vote of align_matches (recognizer.py:222-271, 303-310) for Q
 * queries at once.  Query q owns (hash, offset) pairs [query_starts[q], query_starts[q+1]);
 * duplicates of a (hash, offset) pair inside one query are ignored (the callers pass a
 * set, recognizer.py:378-382).  Per query, up to topn results, best first:
 *   out_song / out_diff  — song id and winning offset difference (db_offset - query_offset;
 *                          smallest difference among equal counts),
 *   out_count            — aligned matches in that bin,
 *   out_rows             — dedup_hashes[song]: DB rows matched, counted once per row,
 *   out_nres[q]          — number of valid results (<= topn).
 * Equal counts order by ascending song id (stable sort, recognizer.py:307-310).
 * The vote is the partitioned vote of csrc/index_pvote.cu (vote tuples written once into per-(query, partition)
 * regions and counted in shared memory); a query it cannot take is voted by per-query hash tables in HBM (any size).
 * h_stats (optional, 4 x int64): query (hash, offset) pairs, DB rows matched (the total of
 * dedup_hashes), (song, diff) tuples voted (len(results) of return_matches), distinct bins. */
int sia_index_query_batch(sia_index *ix, const uint8_t *d_hash, const int32_t *d_qoff,
                          const int64_t *h_query_starts, int32_t n_queries, int32_t topn,
                          int32_t *d_out_song, int32_t *d_out_diff, int32_t *d_out_count,
                          int32_t *d_out_rows, int32_t *d_out_nres, int64_t *h_stats, void *stream);

/* The a-priori early exit of recognizer_apriori.py:246-310 for Q queries at once: each query's distinct hashes are
 * read in batches of batch_hashes, and the query stops after the first batch at which the best song has more than
 * twice the matched DB rows of the runner-up (recognizer_apriori.py:305, in integers: rows(s1) > 2 * rows(s2), at
 * least two songs matched).  Batch k of a query is its distinct hashes [k*B, (k+1)*B) in ASCENDING DIGEST ORDER (the
 * reference iterates a Python set, whose order Python does not define; sorted order makes the result independent
 * of how the caller orders the pairs).  The state after batch k is the vote of sia_index_query_batch over the vote
 * tuples and matched rows of batches 0..k only.  Inputs and the five outputs as sia_index_query_batch, taken at the
 * exit batch (or after the last batch if the rule never fires), plus per query:
 *   out_batches[q] — batches read (0 for an empty query),   out_exit[q] — 1 if the rule fired.
 * The rule always looks at the top two, whatever topn.  batch_hashes >= 1, topn >= 1.
 * h_stats (optional, 4 x int64): query (hash, offset) pairs, DB rows read up to each query's exit, vote tuples read
 * up to each query's exit, batches read in all. */
int sia_index_query_apriori(sia_index *ix, const uint8_t *d_hash, const int32_t *d_qoff, const int64_t *h_query_starts,
                            int32_t n_queries, int32_t topn, int32_t batch_hashes,
                            int32_t *d_out_song, int32_t *d_out_diff, int32_t *d_out_count, int32_t *d_out_rows,
                            int32_t *d_out_nres, int32_t *d_out_batches, int32_t *d_out_exit,
                            int64_t *h_stats, void *stream);

/* device time (ms, CUDA events on the call's stream) of the last sia_index_query_batch or sia_index_query_apriori: [0] pack + sort + lookup,
 * [1] vote (all passes of the call) */
int sia_index_query_timing(const sia_index *ix, double *h_ms2);

/* Vote keys: what the (song_id, offset_difference) tuples of return_matches (recognizer.py:268) look like on the
 * device — 64 bits: head (1) | query id (14) | song id (24) | offset difference + 2^24 (25).  head = 1 marks a tuple
 * that also counts as one matched DB row (dedup_hashes, recognizer.py:259-264: the first query offset of its hash). */
#define SIA_KEY_DIFF_BITS 25
#define SIA_KEY_SONG_BITS 24
#define SIA_KEY_QID_BITS  14
#define SIA_DIFF_BIAS     (1 << 24)

/* The vote of align_matches (recognizer.py:303-310) over n_keys vote keys in any order: same outputs as
 * sia_index_query_batch (out_rows counts the head keys of the winners).  n_queries <= 16384; song ids <= max_song. */
int sia_vote_tuples(int device, const uint64_t *d_key, int64_t n_keys, int32_t n_queries, int32_t topn, int32_t max_song,
                    int32_t *d_out_song, int32_t *d_out_diff, int32_t *d_out_count, int32_t *d_out_rows,
                    int32_t *d_out_nres, void *stream);

/* ---- multi-GPU: hash-prefix sharding (the exchanges themselves are NCCL all-to-alls driven by the host layer) ----
 * One query pass = sia_route_entries on the rank that owns the queries -> all-to-all of the entry slots ->
 * sia_index_expand_slots on the shard that owns the hashes -> all-to-all of the key slots -> sia_vote_key_slots on
 * the queries' owner.  A bin's count is the SUM over shards, so every vote key travels and the result equals the
 * single-index result, tie-breaks included.  Slots have fixed capacities (equal-split all-to-alls, no size
 * negotiation on the host); element 0 of a slot holds its count; overflow is reported, never silent.
 *
 * sia_route_entries: d_slots = world slots of slot_cap 16-byte entries; entry = (global query id = qid_base + local
 * query, hash, query offset); destination = floor(prefix16(hash) * world / 65536).  d_status: int32 flags (2 = offset
 * or query id out of range). */
int sia_route_entries(int device, const uint8_t *d_hash, const int32_t *d_qoff, const int64_t *d_query_starts,
                      int32_t n_queries, int64_t n, int32_t qid_base, int32_t world, int64_t slot_cap, void *d_slots,
                      int32_t *d_status, void *stream);
/* d_entry_slots: the world slots received from all ranks.  Rank r owns the global query ids
 * [r * queries_per_rank, (r + 1) * queries_per_rank).  d_key_slots: world slots of key_cap vote keys (local query ids).
 * d_info (4 x int64, accumulated — zero it before a pass): [0] flags (1 = a received entry slot had overflowed at its
 * sender, 2 = a key slot overflowed), [1] largest key slot size needed, [2] largest entry slot size needed. */
int sia_index_expand_slots(sia_index *ix, const void *d_entry_slots, int32_t world, int64_t entry_cap,
                           int32_t queries_per_rank, uint64_t *d_key_slots, int64_t key_cap, int64_t *d_info,
                           void *stream);
/* defer != 0: return as soon as everything is enqueued on `stream` (the host can then prepare the next pass on another
 * stream while this vote runs); sia_vote_finish(device) waits for it and completes the call — one vote in flight per
 * device, key slots and outputs must stay alive until then. */
int sia_vote_key_slots(int device, const uint64_t *d_key_slots, int32_t n_slots, int64_t key_cap, int32_t n_queries,
                       int32_t topn, int32_t max_song, int32_t *d_out_song, int32_t *d_out_diff, int32_t *d_out_count,
                       int32_t *d_out_rows, int32_t *d_out_nres, int32_t defer, void *stream);
int sia_vote_finish(int device);

/* ---- multi-GPU: the same pass with the second exchange FUSED into the scatter kernel over NVLink peer memory ----
 * Instead of writing vote keys, exchanging them (all-to-all #2) and partitioning them at the query's owner, the shard that
 * owns the hashes scatters the vote tuples of its posting runs straight into the (query, partition) regions of the
 * partitioned vote IN THE OWNER'S MEMORY (peer stores + peer atomicAdd through NVLink); the owner then only counts.
 *   sia_peer_alloc / sia_peer_open      one allocation per rank, mapped by every other rank (CUDA IPC; the 64-byte
 *                                       handles travel through the host layer's all-gather)
 *   sia_index_lookup_slots              received entry slots -> sort + lookup (kept inside the handle) and, per GLOBAL
 *                                       query (rank * queries_per_rank + local), the vote tuples this shard holds
 *   [all-reduce (sum) of the tuple counts: every rank then derives the SAME region layout of every owner; the owner
 *    must have zeroed its fill counters and query flags before it joins this all-reduce]
 *   sia_index_scatter_peers             posting runs -> tuples -> the owners' regions (h_peer_*: world pointers each,
 *                                       entry [rank] = the local buffers); consecutive blocks go to different owners
 *                                       and every shard starts with a different one (an owner's NVLink ingress is
 *                                       never the target of all shards at once)
 *   [barrier: all shards have written]
 *   sia_vote_count_regions              the owner counts its regions: same outputs as sia_vote_key_slots.
 * d_info (4 x int64, zeroed per pass): [0] flags (1 = an entry slot overflowed at its sender, 4 = some owner's regions do
 * not fit region_cap tuple slots / fill_cap regions: nothing was scattered or counted), [1] low word: queries that need
 * the key-exchange path (a bin above 24576 tuples), [2] entry slot size needed, [3] region tuple slots needed. */
int sia_peer_alloc(int device, int64_t bytes, void **d_ptr, uint8_t *h_handle64);
int sia_peer_open(int device, const uint8_t *h_handle64, void **d_ptr);
int sia_peer_close(int device, void *d_ptr);
int sia_peer_free(int device, void *d_ptr);
int sia_index_lookup_slots(sia_index *ix, const void *d_entry_slots, int32_t world, int64_t entry_cap,
                           int32_t queries_per_rank, int64_t *d_tuples, int64_t *d_info, void *stream);
int sia_index_scatter_peers(sia_index *ix, int32_t world, int32_t rank, int32_t queries_per_rank, const int64_t *d_tuples_total,
                            void *const *h_peer_regions, void *const *h_peer_fill, void *const *h_peer_qover,
                            int64_t region_cap, int64_t fill_cap, int64_t *d_info, void *stream);
int sia_vote_count_regions(int device, const int64_t *d_tuples_total, int32_t n_queries, int32_t topn, uint64_t *d_regions,
                           uint32_t *d_fill, uint32_t *d_qover, int64_t region_cap, int64_t fill_cap, int32_t *d_out_song,
                           int32_t *d_out_diff, int32_t *d_out_count, int32_t *d_out_rows, int32_t *d_out_nres,
                           int64_t *d_info, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* SIA_B200_H */
