// K2 — get_2D_peaks (__init__.py:116-177) on the time-major dB spectrogram.
//
//   local_max = maximum_filter(A, footprint) == A           (:143, scipy mode='reflect')
//   eroded_bg = binary_erosion(A == 0, footprint, border=1) (:147-148)
//   peak      = (local_max XOR eroded_bg) and A > amp_min   (:151,161)
//
// For a max filter 'reflect' equals clipping the window to the array, and eroded_bg can
// only be true where the whole clipped window is 0 (then local_max is true as well), so
//   peak = (A == max(window)) and not all(window == 0) and A > amp_min.
// The all-zero term can only matter when amp_min < 0 and is compiled in only then.
//
// Stage 1 writes a bitmap, 1 bit per spectrogram element.  Four kernels:
//   peaks_square_warp_tma_kernel  the pipeline's kernel (float32 dB, square 21x21 = CONNECTIVITY_MASK 2, the reference
//     default, amp_min >= 0): persistent CTAs (4 per SM) walk 64-frame x 96-bin tiles; the 84 x 120 halo tile arrives
//     by one TMA tensor copy (cp.async.bulk.tensor.2d, out-of-range elements arrive as zeros) into one buffer on an
//     mbarrier, the next tile prefetched into L2 meanwhile (cp.async.bulk.prefetch.tensor);
//     each warp owns 16 frames, each lane a float4 column: vertical 21-max in registers (van Herk / Gil-Werman: suffix
//     maxima of one block of rows, prefix maxima of the next, one max to combine), horizontal 21-max across lanes with
//     shuffles; 4 ballots per frame go to a striped bitmap [frame][22 strips][4 words];
//   peaks_square_kernel<T, N, EROSION>  float64 input (the bit-exact parity path) and amp_min < 0: one CTA per
//     64-frame x 128-bin tile + halo in shared memory; the separable filter as a sliding max down the frames with
//     threads along bins, a transposed store, then a sliding max along the bins with threads along frames (register
//     windows, log-doubling); plain bitmap [frame][65 words];
//   peaks_footprint_kernel<T, EROSION>  every other footprint, half-width 1..SIA_MAX_NBHD, square or diamond: halo tile
//     in shared memory, van Herk / Gil-Werman sliding maxima along lines (square: time then bins; diamond: two lattice
//     classes of an antidiagonal then a diagonal pass), the erosion term by the same filter on |A|; plain bitmap;
//   peaks_generic_kernel<T>  the diamond at half-width <= 3 (float32 input) or 1 (float64), brute force: it is faster
//     there (DESIGN §14).
// Stage 2 (peaks_rowcount/extract): bitmap -> per-row popcounts -> scan -> ordered
//   (t asc, f asc) peak lists per track, which is the order generate_hashes' stable
//   sort by time produces (__init__.py:194-195).
#include "sia_common.cuh"
#include "stft.cuh"

#include <cuda.h>
#include <cudaTypedefs.h>
#include <math.h>
#include <math_constants.h>
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <string>

namespace sia {

namespace {

constexpr int kThreads = 256;
constexpr int RC = 16;  // outputs per thread in the sliding passes
constexpr size_t kMaxSmemOptin = 227 * 1024;  // dynamic shared memory one CTA may opt in to (sm_100)

template <typename T> __device__ __forceinline__ T neg_inf();
template <> __device__ __forceinline__ float neg_inf<float>() { return -CUDART_INF_F; }
template <> __device__ __forceinline__ double neg_inf<double>() { return -CUDART_INF; }

// v[0..LEN) -> out[i] = op over v[i .. i+W) for i < OUTN, all indices compile-time
template <typename T, int W, int LEN, int OUTN, bool IS_MAX>
__device__ __forceinline__ void sliding(T (&v)[LEN]) {
  constexpr int P = W >= 16 ? 16 : (W >= 8 ? 8 : (W >= 4 ? 4 : (W >= 2 ? 2 : 1)));
#pragma unroll
  for (int s = 1; s < P; s <<= 1) {
#pragma unroll
    for (int i = 0; i + s < LEN; ++i) v[i] = IS_MAX ? max(v[i], v[i + s]) : min(v[i], v[i + s]);
  }
  if (W > P) {
#pragma unroll
    for (int i = 0; i < OUTN; ++i) {
      T x = v[i + W - P];
      if (W - P > P) {  // W up to 33 = 16 + 17: needs a third term
        T y = v[i + P];
        x = IS_MAX ? max(x, y) : min(x, y);
      }
      v[i] = IS_MAX ? max(v[i], x) : min(v[i], x);
    }
  }
}

// 21-wide window with 3-input max (FMNMX3): 3 -> 9 -> 21, 78 ops per 16 outputs
template <int LEN, int OUTN>
__device__ __forceinline__ void sliding21_max3(float (&v)[LEN]) {
  static_assert(LEN >= OUTN + 20, "window does not fit");
#pragma unroll
  for (int i = 0; i + 2 < LEN; ++i) v[i] = fmaxf(fmaxf(v[i], v[i + 1]), v[i + 2]);          // [i, i+3)
#pragma unroll
  for (int i = 0; i + 8 < LEN; ++i) v[i] = fmaxf(fmaxf(v[i], v[i + 3]), v[i + 6]);          // [i, i+9)
#pragma unroll
  for (int i = 0; i < OUTN; ++i) v[i] = fmaxf(fmaxf(v[i], v[i + 9]), v[i + 12]);             // [i, i+21)
}

// The same 16 windows of 21 out of 36 values, van Herk / Gil-Werman style: suffix maxima of v[0..20], prefix maxima of
// v[21..35], out[i] = max(suffix[i], prefix[i + 20]) — 49 max operations instead of 78 (the two scans advance two
// elements per step with a 3-input max, so the dependent chains are 10 and 7 long).
__device__ __forceinline__ void vanherk21_36(float (&v)[36]) {
  // suffix: v[i] = max(v[i..20]), i = 19 .. 0
#pragma unroll
  for (int i = 18; i >= 0; i -= 2) {
    const float s2 = v[i + 2];
    const float a = fmaxf(v[i + 1], s2);
    v[i] = fmaxf(fmaxf(v[i], v[i + 1]), s2);
    v[i + 1] = a;
  }
  // prefix: v[j] = max(v[21..j]), j = 22 .. 35
#pragma unroll
  for (int j = 22; j + 1 <= 35; j += 2) {
    const float p2 = v[j - 1];
    const float a = fmaxf(v[j], p2);
    v[j + 1] = fmaxf(fmaxf(v[j + 1], v[j]), p2);
    v[j] = a;
  }
#pragma unroll
  for (int i = 1; i < 16; ++i) v[i] = fmaxf(v[i], v[i + 20]);
}

struct TileCoord {
  int trk;
  int64_t row_lo, row_hi;  // global rows of this track [row_lo, row_hi)
  int64_t r0;              // first output row (global) of the tile
  int f0;                  // first output bin of the tile
};

__device__ __forceinline__ TileCoord tile_coord(const int64_t *__restrict__ frame_starts,
                                                const int64_t *__restrict__ ttile_starts, int n_tracks) {
  constexpr int kFTiles = (SIA_NBINS + kPeakTileF - 1) / kPeakTileF;  // 17
  TileCoord tc;
  const int64_t tt = blockIdx.x / kFTiles;
  tc.f0 = (int)(blockIdx.x % kFTiles) * kPeakTileF;
  tc.trk = find_segment(ttile_starts, n_tracks, tt);
  tc.row_lo = frame_starts[tc.trk];
  tc.row_hi = frame_starts[tc.trk + 1];
  tc.r0 = tc.row_lo + (tt - ttile_starts[tc.trk]) * kPeakTileT;
  return tc;
}

// Load the (TT+2N) x (TF+2N) halo tile; out-of-track rows and out-of-range bins get `fill`.
template <typename T, int N, int AS>
__device__ __forceinline__ void load_tile(T *__restrict__ A, const T *__restrict__ spec, const TileCoord &tc, T fill) {
  constexpr int ROWS = kPeakTileT + 2 * N, COLS = kPeakTileF + 2 * N;
  for (int idx = threadIdx.x; idx < ROWS * COLS; idx += kThreads) {
    const int r = idx / COLS, c = idx - r * COLS;
    const int64_t g = tc.r0 - N + r;
    const int f = tc.f0 - N + c;
    T v = fill;
    if (g >= tc.row_lo && g < tc.row_hi && f >= 0 && f < SIA_NBINS) v = spec[g * SIA_F_STRIDE + f];
    A[r * AS + c] = v;
  }
}

// ---- fast path: square footprint, compile-time half-width N -------------------------------------
template <typename T, int N, bool EROSION>
__global__ void __launch_bounds__(kThreads)
peaks_square_kernel(const T *__restrict__ spec, const int64_t *__restrict__ frame_starts,
                    const int64_t *__restrict__ ttile_starts, int n_tracks, double amp_min,
                    uint32_t *__restrict__ bitmap) {
  constexpr int TT = kPeakTileT, TF = kPeakTileF;
  constexpr int ROWS = TT + 2 * N, COLS = TF + 2 * N;
  constexpr int AS = COLS | 1;     // odd row stride: column walks with threads along rows are conflict-free
  constexpr int VS = TT + 1;       // odd stride of the transposed intermediate
  constexpr int W = 2 * N + 1, LEN = RC + 2 * N;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T *A = reinterpret_cast<T *>(smem_raw);            // [ROWS][AS]
  T *VT = A + ROWS * AS;                             // [COLS][VS]   max down the rows, transposed
  T *VTmin = VT + COLS * VS;                         // [COLS][VS]   (EROSION only)
  uint16_t *sbits = reinterpret_cast<uint16_t *>(EROSION ? (VTmin + COLS * VS) : VTmin);  // [TT][TF/16]

  const TileCoord tc = tile_coord(frame_starts, ttile_starts, n_tracks);
  load_tile<T, N, AS>(A, spec, tc, neg_inf<T>());
  __syncthreads();

  // pass V: thread = (bin column c, row chunk q); window slides down the rows
  for (int task = threadIdx.x; task < COLS * (TT / RC); task += kThreads) {
    const int q = task / COLS, c = task - q * COLS;
    T v[LEN];
#pragma unroll
    for (int i = 0; i < LEN; ++i) v[i] = A[(q * RC + i) * AS + c];
    if (EROSION) {
      T u[LEN];
#pragma unroll
      for (int i = 0; i < LEN; ++i) u[i] = v[i] == neg_inf<T>() ? -neg_inf<T>() : v[i];  // outside: +inf for min
      sliding<T, W, LEN, RC, false>(u);
#pragma unroll
      for (int i = 0; i < RC; ++i) VTmin[c * VS + q * RC + i] = u[i];
    }
    sliding<T, W, LEN, RC, true>(v);
#pragma unroll
    for (int i = 0; i < RC; ++i) VT[c * VS + q * RC + i] = v[i];
  }
  __syncthreads();

  // pass H: thread = (frame row r, bin chunk j); window slides along the bins
  for (int task = threadIdx.x; task < TT * (TF / RC); task += kThreads) {
    const int j = task / TT, r = task - j * TT;
    T v[LEN];
#pragma unroll
    for (int i = 0; i < LEN; ++i) v[i] = VT[(j * RC + i) * VS + r];
    sliding<T, W, LEN, RC, true>(v);
    T u[LEN];
    if (EROSION) {
#pragma unroll
      for (int i = 0; i < LEN; ++i) u[i] = VTmin[(j * RC + i) * VS + r];
      sliding<T, W, LEN, RC, false>(u);
    }
    const bool row_ok = tc.r0 + r < tc.row_hi;
    uint32_t bits = 0;
#pragma unroll
    for (int i = 0; i < RC; ++i) {
      const T ctr = A[(r + N) * AS + j * RC + i + N];
      bool pk = row_ok && (tc.f0 + j * RC + i < SIA_NBINS) && ctr == v[i] && (double)ctr > amp_min;
      if (EROSION) pk = pk && !(v[i] == (T)0 && u[i] == (T)0);
      bits |= (uint32_t)pk << i;
    }
    sbits[r * (TF / 16) + j] = (uint16_t)bits;
  }
  __syncthreads();

  // bitmap words: TT rows x TF/32 words per tile
  for (int idx = threadIdx.x; idx < TT * (TF / 32); idx += kThreads) {
    const int r = idx / (TF / 32), w = idx - r * (TF / 32);
    const int64_t g = tc.r0 + r;
    const int gw = tc.f0 / 32 + w;
    if (g < tc.row_hi && gw < SIA_ROW_WORDS) {
      const uint32_t word = (uint32_t)sbits[r * (TF / 16) + 2 * w] | ((uint32_t)sbits[r * (TF / 16) + 2 * w + 1] << 16);
      bitmap[g * kBitmapRowWords + gw] = word;
    }
  }
}

// ---- production path: float32, square 21x21, amp_min >= 0 ------------------------------------------------
// One CTA = 64 frames x 96 bins (3 bitmap words per frame); 4 warps, warp q owns frames 16q..16q+15.
// The 84 x 120 halo tile is staged in shared memory as float4.  Each lane owns one float4 column: it slides
// the 21-frame max down its 4 bins entirely in registers (van Herk, two bins at a time), then takes the
// 21-bin max across lanes with 10 shuffles of per-lane prefix / suffix / block maxima — no second
// shared-memory pass, no transposes.  Lanes 0..23 produce the 96
// outputs, lanes 24..29 carry the +-12-bin halo columns, lanes 30..31 idle.
constexpr int kW2Rows = kPeakTileT;                                 // 64
constexpr int kW2Bins = 96;
constexpr int kW2Cols4 = 30;                                        // (96 + 2*12) / 4
constexpr int kW2Strips = (SIA_NBINS + kW2Bins - 1) / kW2Bins;      // 22
constexpr int kW2Threads = 128;
constexpr int kW2TileRows = kW2Rows + 20;                           // 84

// The filter proper, on a staged tile A (84 x 30 float4): see the kernel comment above.
__device__ __forceinline__ void warp_tile_peaks(const float4 *__restrict__ A, uint32_t a_base, int64_t r0, int64_t row_hi,
                                                int strip, int f0, float amp_lo, uint32_t *__restrict__ bitmap) {
  const int lane = threadIdx.x & 31, q = threadIdx.x >> 5;
  const int col = lane < kW2Cols4 ? (lane + 3) % kW2Cols4 : 0;      // lanes 0..23 -> columns 3..26 (outputs)
  auto src = [&](int k) { return lane < kW2Cols4 ? (lane + k + kW2Cols4) % kW2Cols4 : lane; };
  const int s_m1 = src(-1), s_m2 = src(-2), s_m3 = src(-3), s_p1 = src(1), s_p2 = src(2), s_p3 = src(3);

  // the vertical pass one half of the column at a time (bins 0,1 then 2,3): 72 values in flight instead of 144, so
  // the kernel fits the registers of kW2CtasPerSM resident CTAs
  float vx[36], vy[36], vz[36], vw[36];
  const float2 *A2 = reinterpret_cast<const float2 *>(A);
#pragma unroll
  for (int i = 0; i < 36; ++i) {
    const float2 t = A2[2 * ((16 * q + i) * kW2Cols4 + col)];
    vx[i] = t.x; vy[i] = t.y;
  }
  vanherk21_36(vx);
  vanherk21_36(vy);
#pragma unroll
  for (int i = 0; i < 36; ++i) {
    const float2 t = A2[2 * ((16 * q + i) * kW2Cols4 + col) + 1];
    vz[i] = t.x; vw[i] = t.y;
  }
  vanherk21_36(vz);
  vanherk21_36(vw);

  const unsigned FULL = 0xffffffffu;
  const float amp_up = nextafterf(amp_lo, CUDART_INF_F);
  const int64_t g0 = r0 + 16 * q;                                   // first output frame of this warp
  const int nvalid = (int)min((int64_t)16, row_hi - g0);            // frames of the chunk inside the track
  const int fl = f0 + 4 * lane;
  const bool v0 = lane < 24 && fl < SIA_NBINS, v1 = lane < 24 && fl + 1 < SIA_NBINS;
  const bool v2 = lane < 24 && fl + 2 < SIA_NBINS, v3 = lane < 24 && fl + 3 < SIA_NBINS;
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    const float a0 = vx[i], a1 = vy[i], a2 = vz[i], a3 = vw[i];
    // amp_up (the smallest float above the threshold) rides in the block maximum M, which every window
    // includes, so "centre == window max and centre > amp_min" becomes the single test centre >= h
    const float S2 = fmaxf(a2, a3), S1 = fmaxf(a1, S2), M = fmaxf(fmaxf(a0, S1), amp_up);
    const float P1 = fmaxf(a0, a1), P2 = fmaxf(P1, a2);
    const float Mm1 = __shfl_sync(FULL, M, s_m1), Mp1 = __shfl_sync(FULL, M, s_p1);
    const float Mm2 = __shfl_sync(FULL, M, s_m2), Mp2 = __shfl_sync(FULL, M, s_p2);
    const float S1m2 = __shfl_sync(FULL, S1, s_m2);
    const float S2m3 = __shfl_sync(FULL, S2, s_m3), S3m3 = __shfl_sync(FULL, a3, s_m3);
    const float P2p2 = __shfl_sync(FULL, P2, s_p2);
    const float P0p3 = __shfl_sync(FULL, a0, s_p3), P1p3 = __shfl_sync(FULL, P1, s_p3);
    const float common = fmaxf(fmaxf(Mm1, M), Mp1);
    const float cl = fmaxf(common, Mm2);
    const float h0 = fmaxf(cl, fmaxf(S2m3, P2p2));          // bins -10..+10 around element 0
    const float h1 = fmaxf(cl, fmaxf(S3m3, Mp2));
    const float h2 = fmaxf(cl, fmaxf(Mp2, P0p3));
    const float h3 = fmaxf(fmaxf(common, S1m2), fmaxf(Mp2, P1p3));
    // re-read the centre row from shared memory (volatile: keeps 16 float4 out of the register file)
    float4 c;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];\n"
                 : "=f"(c.x), "=f"(c.y), "=f"(c.z), "=f"(c.w)
                 : "r"(a_base + (uint32_t)((16 * q + i + 10) * kW2Cols4 + col) * 16u));
    // one ballot per element index: word e, bit l  <->  bin f0 + 4*l + e   (striped bitmap layout)
    const uint32_t b0 = __ballot_sync(FULL, c.x >= h0 && v0);
    const uint32_t b1 = __ballot_sync(FULL, c.y >= h1 && v1);
    const uint32_t b2 = __ballot_sync(FULL, c.z >= h2 && v2);
    const uint32_t b3 = __ballot_sync(FULL, c.w >= h3 && v3);
    if (lane == 0 && i < nvalid)
      *reinterpret_cast<uint4 *>(bitmap + (g0 + i) * kBitmapRowWords + 4 * strip) = make_uint4(b0, b1, b2, b3);
  }
}

// Persistent kernel: 4 CTAs per SM walk the tiles with a stride of the grid, one tile buffer each.  The next tile is
// prefetched into L2 while the current one is filtered, and copied into the buffer once the buffer is free.  One
// buffer (41 KB) instead of two lets 4 CTAs = 16 warps share an SM instead of 2 CTAs = 8 warps, which hides the
// latency of the filter's dependent max / shuffle chains; the copy waits of one CTA are covered by the other three.
constexpr int kW2CtasPerSM = 4;
constexpr size_t kW2TileBytes = sizeof(float4) * kW2TileRows * kW2Cols4;
constexpr size_t kW2PersistSmem = kW2TileBytes + 128;

__global__ void __launch_bounds__(kW2Threads, kW2CtasPerSM)
peaks_square_warp_tma_kernel(const int64_t *__restrict__ frame_starts, const int64_t *__restrict__ ttile_starts, int n_tracks,
                             int64_t n_tiles, float amp_lo, uint32_t *__restrict__ bitmap,
                             const __grid_constant__ CUtensorMap tmap) {
  extern __shared__ __align__(128) unsigned char w2_smem[];
  float4 *A = reinterpret_cast<float4 *>(w2_smem);
  unsigned long long *bar = reinterpret_cast<unsigned long long *>(w2_smem + kW2TileBytes);
  const uint32_t bar0 = (uint32_t)__cvta_generic_to_shared(bar);
  const uint32_t base0 = (uint32_t)__cvta_generic_to_shared(w2_smem);
  if (threadIdx.x == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;\n" ::"r"(bar0));
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  }
  __syncthreads();
  // tensor coordinates (first bin, first frame) of the halo tile of `tile`
  auto coords = [&](int64_t tile, int &x, int &y) {
    const int64_t tt = tile / kW2Strips;
    const int strip = (int)(tile - tt * kW2Strips);
    const int trk = find_segment(ttile_starts, n_tracks, tt);
    x = strip * kW2Bins - 12;
    y = (int)(frame_starts[trk] + (tt - ttile_starts[trk]) * kW2Rows - 10);
  };
  // thread 0: start the tensor copy of tile `tile` into the buffer
  auto issue = [&](int64_t tile) {
    int x, y;
    coords(tile, x, y);
    asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");   // earlier generic writes (zeroed frames) vs the copy
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(bar0), "r"((uint32_t)kW2TileBytes)
                 : "memory");
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];\n"
                 ::"r"(base0), "l"(reinterpret_cast<uint64_t>(&tmap)), "r"(x), "r"(y), "r"(bar0) : "memory");
  };
  int64_t tile = blockIdx.x;
  if (threadIdx.x == 0 && tile < n_tiles) issue(tile);
  for (int k = 0; tile < n_tiles; tile += gridDim.x, ++k) {
    const bool has_next = tile + gridDim.x < n_tiles;
    if (threadIdx.x == 0 && has_next) {
      int x, y;
      coords(tile + gridDim.x, x, y);
      asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global.tile [%0, {%1, %2}];\n"
                   ::"l"(reinterpret_cast<uint64_t>(&tmap)), "r"(x), "r"(y) : "memory");
    }
    const int64_t tt = tile / kW2Strips;
    const int strip = (int)(tile - tt * kW2Strips);
    const int trk = find_segment(ttile_starts, n_tracks, tt);
    const int64_t row_lo = frame_starts[trk], row_hi = frame_starts[trk + 1];
    const int64_t r0 = row_lo + (tt - ttile_starts[trk]) * kW2Rows;
    asm volatile("{\n.reg .pred P1;\nLAB_WAIT:\nmbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n@P1 bra DONE;\nbra LAB_WAIT;\nDONE:\n}\n"
                 ::"r"(bar0), "r"(k & 1) : "memory");
    const int64_t g_first = r0 - 10;
    if (g_first < row_lo || g_first + kW2TileRows > row_hi) {      // first / last tiles of a track: zero the other tracks' frames
      for (int i = threadIdx.x; i < kW2TileRows * kW2Cols4; i += kW2Threads) {
        const int64_t g = g_first + i / kW2Cols4;
        if (g < row_lo || g >= row_hi) A[i] = make_float4(0.f, 0.f, 0.f, 0.f);
      }
      __syncthreads();
    }
    warp_tile_peaks(A, base0, r0, row_hi, strip, strip * kW2Bins, amp_lo, bitmap);
    __syncthreads();                                               // every warp is done with the buffer
    if (threadIdx.x == 0 && has_next) issue(tile + gridDim.x);
  }
}

// tensor map of the chunk's spectrogram for the TMA tile loads: [total_frames][2049] float32, row pitch 2080 floats,
// box = one halo tile (84 frames x 120 bins), zero fill outside
int make_spec_tensor_map(const float *spec, int64_t total_frames, CUtensorMap *tm) {
  static PFN_cuTensorMapEncodeTiled encode = nullptr;
  if (!encode) {
    cudaDriverEntryPointQueryResult qres;
    void *fn = nullptr;
    SIA_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
    SIA_REQUIRE(fn != nullptr && qres == cudaDriverEntryPointSuccess, SIA_E_CUDA, "cuTensorMapEncodeTiled is not available");
    encode = reinterpret_cast<PFN_cuTensorMapEncodeTiled>(fn);
  }
  const cuuint64_t gdim[2] = {(cuuint64_t)SIA_NBINS, (cuuint64_t)total_frames};
  const cuuint64_t gstride[1] = {(cuuint64_t)SIA_F_STRIDE * sizeof(float)};
  const cuuint32_t box[2] = {(cuuint32_t)(4 * kW2Cols4), (cuuint32_t)kW2TileRows};
  const cuuint32_t estride[2] = {1, 1};
  const CUresult r = encode(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float *>(spec), gdim, gstride, box, estride,
                            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  SIA_REQUIRE(r == CUDA_SUCCESS, SIA_E_CUDA, "cuTensorMapEncodeTiled failed for the spectrogram");
  return SIA_OK;
}

int launch_square_warp(const PeaksLaunch &a, cudaStream_t s) {
  // float c > (double) amp_min  <=>  c > amp_lo with amp_lo = amp_min rounded DOWN to float
  float amp_lo = (float)a.amp_min;
  if ((double)amp_lo > a.amp_min) amp_lo = nextafterf(amp_lo, -INFINITY);
  const int64_t blocks = a.total_ttiles * kW2Strips;
  alignas(64) CUtensorMap tm;
  memset(&tm, 0, sizeof tm);
  int rc = make_spec_tensor_map((const float *)a.d_spec, a.total_frames, &tm);
  if (rc) return rc;
  SIA_CUDA(cudaFuncSetAttribute(peaks_square_warp_tma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kW2PersistSmem));
  const unsigned grid = (unsigned)std::min<int64_t>(blocks, kW2CtasPerSM * kNumSMs);
  peaks_square_warp_tma_kernel<<<grid, kW2Threads, kW2PersistSmem, s>>>(a.d_frame_starts, a.d_ttile_starts, a.n_tracks, blocks,
                                                                        amp_lo, a.d_bitmap, tm);
  SIA_CHECK_LAUNCH();
  return SIA_OK;
}

// ---- footprint-general path: any half-width r in 1..SIA_MAX_NBHD, square or diamond ------------------------------
// van Herk / Gil-Werman sliding max along one line: out[k] = max(in[k .. k+W-1]) for the outputs k of block q,
// [q*W, min(q*W + W, n)); in[] holds n + W - 1 values.  Suffix maxima of block q, then prefix maxima of block q+1
// combined into the outputs: about 3 max operations per output whatever W is.  ACC folds the result into out[].
template <typename T, bool ACC>
__device__ __forceinline__ void vh_block(const T *__restrict__ in, int is, T *__restrict__ out, int os, int n, int W,
                                         int q) {
  const int k0 = q * W;
  T s = neg_inf<T>();
  for (int k = k0 + W - 1; k >= k0; --k) {
    s = max(s, in[k * is]);
    if (k < n) out[k * os] = ACC ? max(out[k * os], s) : s;
  }
  T p = neg_inf<T>();
  const int jend = min(k0 + 2 * W - 1, n + W - 1);
  for (int j = k0 + W; j < jend; ++j) {
    p = max(p, in[j * is]);
    out[(j - W + 1) * os] = max(out[(j - W + 1) * os], p);
  }
}

// Shared-memory shape of one footprint tile: TT output frames x TF output bins (TF a multiple of 32), halo r.
//   A  [TT+2r][(TF+2r)|1]  the spectrogram around the tile, -inf outside the track and outside bins 0..2048
//   I  square: [TT][(TF+2r)|1] max along time;  diamond: [TT+r][(TF+r)|1] max along one antidiagonal segment
//   M  [TT][TF+1]           the window maximum
//   bits [TT][TF/32]
struct FootprintTile {
  int r, tt, tf;
  bool diamond;
  __host__ __device__ int a_stride() const { return (tf + 2 * r) | 1; }
  __host__ __device__ int i_rows() const { return diamond ? tt + r : tt; }
  __host__ __device__ int i_stride() const { return diamond ? (tf + r) | 1 : a_stride(); }
  size_t smem(size_t elem) const {
    const size_t vals = (size_t)(tt + 2 * r) * a_stride() + (size_t)i_rows() * i_stride() + (size_t)tt * (tf + 1);
    return vals * elem + (size_t)tt * (tf / 32) * sizeof(uint32_t);
  }
};

constexpr int kFpThreads = 512;

// Reached from r = 2 on float64 input and from r = 4 on float32: smaller diamonds take the brute-force kernel.
// The L1 ball |dt| + |df| <= r is, in the rotated coordinates u = dt + df, v = dt - df, the square max(|u|, |v|) <= r
// on the lattice u = v (mod 2).  Its even class (u, v even) is {(i+j, i-j) : i, j in [-k0, k0]}, k0 = floor(r/2),
// and its odd class {(1+i+j, i-j) : i, j in [-k1, k1-1]}, k1 = floor((r+1)/2): each a Minkowski sum of one segment
// along the antidiagonal (1,-1) and one along the diagonal (1,1), of r+1 and r points (in either order).  So the
// diamond max is the larger of two separable maxima, antidiagonal pass first (D1) then diagonal pass (D2).  D1 is
// evaluated on every position its diagonal segments reach, also outside the track or the bin range: such a
// position takes the max of the in-range points of its segment (the rest are -inf in A), so the clipped window is
// exact near every border.
template <typename T>
__device__ __forceinline__ void diamond_class(const T *__restrict__ A, T *__restrict__ B, T *__restrict__ M,
                                              const FootprintTile &g, int odd) {
  const int r = g.r, TT = g.tt, TF = g.tf, AS = g.a_stride(), BS = g.i_stride(), MS = TF + 1;
  const int kk = odd ? (r + 1) / 2 : r / 2;
  const int Wc = odd ? 2 * kk : 2 * kk + 1;  // segment length
  const int a = -kk, ct = odd;               // segment offsets a .. a+Wc-1; odd class shifted one frame
  const int pt0 = a + ct, BR = TT + Wc - 1, BC = TF + Wc - 1;   // D1 positions: frames pt0.., bins a.. (tile-local)
  // D1: B(p) = max_k A(p_t + a + k, p_f - a - k).  Line u = p_t + p_f, window start at A row m = p_t + a.
  {
    const int u0 = pt0 + a, nu = BR + BC - 1;
    const int nq = (min(BR, BC) + Wc - 1) / Wc;
    for (int task = threadIdx.x; task < nu * nq; task += blockDim.x) {
      const int q = task / nu, u = u0 + (task - q * nu);
      const int m_lo = max(pt0 + a, u - BC + 1), m_hi = min(pt0 + a + BR, u + 1);
      const int n = m_hi - m_lo;
      if (q * Wc >= n) continue;
      vh_block<T, false>(A + (m_lo + r) * AS + (u - m_lo + r), AS - 1, B + (m_lo - a - pt0) * BS + (u - m_lo), BS - 1,
                         n, Wc, q);
    }
  }
  __syncthreads();
  // D2: M(t, f) = max(M, max_k B(t + k, f + k)) in B's own coordinates, along the diagonals d = f - t
  {
    const int nd = TT + TF - 1;
    const int nq = (min(TT, TF) + Wc - 1) / Wc;
    for (int task = threadIdx.x; task < nd * nq; task += blockDim.x) {
      const int q = task / nd, d = task - q * nd - (TT - 1);
      const int t_lo = max(0, -d), n = min(TT, TF - d) - t_lo;
      if (q * Wc >= n) continue;
      if (odd) vh_block<T, true>(B + t_lo * BS + t_lo + d, BS + 1, M + t_lo * MS + t_lo + d, MS + 1, n, Wc, q);
      else vh_block<T, false>(B + t_lo * BS + t_lo + d, BS + 1, M + t_lo * MS + t_lo + d, MS + 1, n, Wc, q);
    }
  }
  __syncthreads();
}

// One CTA per 64-frame time tile x TF bins; it walks the time tile in sub-tiles of TT frames.  Per sub-tile:
// stage A, filter (square: time pass then bin pass; diamond: two classes of D1 + D2), compare the centre with M.
// EROSION (amp_min < 0) stages |A| in a second round and runs the same filter: the window is all zero iff
// max |A| == 0 there.
template <typename T, bool EROSION>
__global__ void __launch_bounds__(kFpThreads)
peaks_footprint_kernel(const T *__restrict__ spec, const int64_t *__restrict__ frame_starts,
                       const int64_t *__restrict__ ttile_starts, int n_tracks, double amp_min, const FootprintTile g,
                       uint32_t *__restrict__ bitmap) {
  const int r = g.r, TT = g.tt, TF = g.tf, AS = g.a_stride(), IS = g.i_stride(), MS = TF + 1, WPR = TF / 32;
  const int AR = TT + 2 * r, AC = TF + 2 * r, W = 2 * r + 1;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T *A = reinterpret_cast<T *>(smem_raw);
  T *I = A + (size_t)AR * AS;
  T *M = I + (size_t)g.i_rows() * IS;
  uint32_t *bits = reinterpret_cast<uint32_t *>(M + (size_t)TT * MS);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;

  const int nft = (SIA_NBINS + TF - 1) / TF;
  const int64_t tt = blockIdx.x / nft;
  const int f0 = (int)(blockIdx.x - tt * nft) * TF;
  const int trk = find_segment(ttile_starts, n_tracks, tt);
  const int64_t row_lo = frame_starts[trk], row_hi = frame_starts[trk + 1];
  const int64_t rt = row_lo + (tt - ttile_starts[trk]) * kPeakTileT;

  for (int sub = 0; sub < kPeakTileT; sub += TT) {
    const int64_t r0 = rt + sub;
    if (r0 >= row_hi) break;
    for (int round = 0; round < (EROSION ? 2 : 1); ++round) {
      for (int i = warp; i < AR; i += nwarps) {
        const int64_t gr = r0 - r + i;
        const bool row_ok = gr >= row_lo && gr < row_hi;
        for (int j = lane; j < AC; j += 32) {
          const int f = f0 - r + j;
          T v = neg_inf<T>();
          if (row_ok && f >= 0 && f < SIA_NBINS) {
            v = spec[gr * SIA_F_STRIDE + f];
            if (round && v < (T)0 && v != neg_inf<T>()) v = -v;   // -inf stays 'outside', as in the other kernels
          }
          A[i * AS + j] = v;
        }
      }
      __syncthreads();
      if (!g.diamond) {
        const int nq = (TT + W - 1) / W;
        for (int task = threadIdx.x; task < AC * nq; task += blockDim.x) {   // along time, thread = bin column
          const int q = task / AC, c = task - q * AC;
          vh_block<T, false>(A + c, AS, I + c, IS, TT, W, q);
        }
        __syncthreads();
        const int nq2 = (TF + W - 1) / W;
        for (int task = threadIdx.x; task < TT * nq2; task += blockDim.x) {  // along bins, thread = frame row
          const int q = task / TT, t = task - q * TT;
          vh_block<T, false>(I + t * IS, 1, M + t * MS, 1, TF, W, q);
        }
        __syncthreads();
      } else {
        diamond_class<T>(A, I, M, g, 0);
        diamond_class<T>(A, I, M, g, 1);
      }
      for (int t = warp; t < TT; t += nwarps) {
        const bool row_ok = r0 + t < row_hi;
        for (int w = 0; w < WPR; ++w) {
          const int c = 32 * w + lane;
          if (round == 0) {
            const T ctr = A[(t + r) * AS + c + r];
            const bool pk = row_ok && f0 + c < SIA_NBINS && ctr == M[t * MS + c] && (double)ctr > amp_min;
            const uint32_t word = __ballot_sync(0xffffffffu, pk);
            if (lane == 0) bits[t * WPR + w] = word;
          } else {
            const uint32_t zero = __ballot_sync(0xffffffffu, M[t * MS + c] == (T)0);
            if (lane == 0) bits[t * WPR + w] &= ~zero;
          }
        }
      }
      __syncthreads();
    }
    for (int idx = threadIdx.x; idx < TT * WPR; idx += blockDim.x) {
      const int t = idx / WPR, w = idx - t * WPR;
      const int gw = f0 / 32 + w;
      if (r0 + t < row_hi && gw < SIA_ROW_WORDS) bitmap[(r0 + t) * kBitmapRowWords + gw] = bits[idx];
    }
  }
}

// The tile shape for (element size, r, footprint): the largest share of output bins among the staged ones that fits
// one CTA's shared memory.
FootprintTile footprint_tile(size_t elem, int r, bool diamond) {
  FootprintTile best{r, 0, 0, diamond};
  double best_eff = -1.0;
  for (int tf : {128, 64, 32})
    for (int tt = kPeakTileT; tt >= 1; tt /= 2) {
      const FootprintTile g{r, tt, tf, diamond};
      if (g.smem(elem) > (size_t)kMaxSmemOptin) continue;
      const double eff = (double)tt * tf / ((double)(tt + 2 * r) * (tf + 2 * r));
      if (eff > best_eff) { best_eff = eff; best = g; }
    }
  return best;
}

template <typename T, bool E>
int launch_footprint(const PeaksLaunch &a, cudaStream_t s) {
  const FootprintTile g = footprint_tile(sizeof(T), a.nbhd, a.connectivity == 1);
  SIA_REQUIRE(g.tt > 0, SIA_E_UNSUPPORTED, "peaks: no footprint tile fits shared memory");
  const size_t smem = g.smem(sizeof(T));
  auto kern = peaks_footprint_kernel<T, E>;
  SIA_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int64_t blocks = a.total_ttiles * ((SIA_NBINS + g.tf - 1) / g.tf);
  kern<<<(unsigned)blocks, kFpThreads, smem, s>>>((const T *)a.d_spec, a.d_frame_starts, a.d_ttile_starts, a.n_tracks,
                                                 a.amp_min, g, a.d_bitmap);
  SIA_CHECK_LAUNCH();
  return SIA_OK;
}

// ---- brute force: the diamond at small half-widths, where it is faster than the footprint kernel ----
// Measured (DESIGN §14): faster at nbhd 1 and 3 on float32 input, at nbhd 1 only on float64.
constexpr int kBruteMaxNbhd = 3;
inline int brute_max_nbhd(int in_type) { return in_type == SIA_F64 ? 1 : kBruteMaxNbhd; }

template <typename T>
__global__ void __launch_bounds__(kThreads)
peaks_generic_kernel(const T *__restrict__ spec, const int64_t *__restrict__ frame_starts,
                     const int64_t *__restrict__ ttile_starts, int n_tracks, double amp_min, int nb, int diamond,
                     int erosion, uint32_t *__restrict__ bitmap) {
  constexpr int TT = kPeakTileT, TF = kPeakTileF, N = kBruteMaxNbhd;
  constexpr int ROWS = TT + 2 * N, COLS = TF + 2 * N;
  constexpr int AS = COLS | 1;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T *A = reinterpret_cast<T *>(smem_raw);

  const TileCoord tc = tile_coord(frame_starts, ttile_starts, n_tracks);
  load_tile<T, N, AS>(A, spec, tc, neg_inf<T>());
  __syncthreads();

  for (int idx = threadIdx.x; idx < TT * TF; idx += kThreads) {   // warp = 32 consecutive bins of one frame
    const int r = idx / TF, c = idx - r * TF;
    const int64_t g = tc.r0 + r;
    const int f = tc.f0 + c;
    const T ctr = A[(r + N) * AS + c + N];
    bool pk = g < tc.row_hi && f < SIA_NBINS && (double)ctr > amp_min;
    if (pk) {
      bool allzero = true;
      for (int dt = -nb; dt <= nb && pk; ++dt) {
        const int wf = diamond ? nb - abs(dt) : nb;
        const T *rowp = A + (r + N + dt) * AS + c + N;
        for (int df = -wf; df <= wf; ++df) {
          const T x = rowp[df];
          if (x > ctr) { pk = false; break; }
          if (x != (T)0 && x != neg_inf<T>()) allzero = false;
        }
      }
      if (erosion && allzero) pk = false;
    }
    const uint32_t word = __ballot_sync(0xffffffffu, pk);
    const int gw = f >> 5;
    if ((threadIdx.x & 31) == 0 && g < tc.row_hi && gw < SIA_ROW_WORDS) bitmap[g * kBitmapRowWords + gw] = word;
  }
}

template <typename T, int N, bool E>
int launch_square(const PeaksLaunch &a, cudaStream_t s) {
  constexpr int ROWS = kPeakTileT + 2 * N, COLS = kPeakTileF + 2 * N, AS = COLS | 1, VS = kPeakTileT + 1;
  const size_t smem = sizeof(T) * (ROWS * AS + COLS * VS * (E ? 2 : 1)) + kPeakTileT * (kPeakTileF / 16) * 2;
  auto kern = peaks_square_kernel<T, N, E>;
  SIA_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int64_t blocks = a.total_ttiles * ((SIA_NBINS + kPeakTileF - 1) / kPeakTileF);
  kern<<<(unsigned)blocks, kThreads, smem, s>>>((const T *)a.d_spec, a.d_frame_starts, a.d_ttile_starts, a.n_tracks,
                                              a.amp_min, a.d_bitmap);
  SIA_CHECK_LAUNCH();
  return SIA_OK;
}

template <typename T>
int launch_generic(const PeaksLaunch &a, cudaStream_t s) {
  constexpr int N = kBruteMaxNbhd;
  constexpr int ROWS = kPeakTileT + 2 * N, COLS = kPeakTileF + 2 * N, AS = COLS | 1;
  const size_t smem = sizeof(T) * ROWS * AS;
  auto kern = peaks_generic_kernel<T>;
  SIA_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int64_t blocks = a.total_ttiles * ((SIA_NBINS + kPeakTileF - 1) / kPeakTileF);
  kern<<<(unsigned)blocks, kThreads, smem, s>>>((const T *)a.d_spec, a.d_frame_starts, a.d_ttile_starts, a.n_tracks,
                                              a.amp_min, a.nbhd, a.connectivity == 1, a.amp_min < 0, a.d_bitmap);
  SIA_CHECK_LAUNCH();
  return SIA_OK;
}

// ---- stage 2 ------------------------------------------------------------------------------------------
// Two bitmap layouts, both with a row stride of kBitmapRowWords words:
//   plain   : word w, bit b            <-> bin 32*w + b              (65 words; tile / generic kernels)
//   striped : word 4*s + e, bit l      <-> bin 96*s + 4*l + e        (22 strips x 4 words; warp kernel)
// WIN (streaming): rows outside their segment's emit window count 0 and yield nothing (PeakWindow, stft.cuh)
__device__ __forceinline__ bool row_in_window(const PeakWindow &w, int64_t g, int &seg, int64_t &k) {
  seg = find_segment(w.frame_starts, w.n, g);
  k = g - w.frame_starts[seg];
  return k >= w.emit_lo[seg] && k < w.emit_hi[seg];
}

template <bool STRIPED, bool WIN>
__global__ void __launch_bounds__(256)
rowcount_kernel(const uint32_t *__restrict__ bitmap, int64_t total_frames, uint32_t *__restrict__ row_count,
                const PeakWindow win) {
  const int lane = threadIdx.x & 31;
  const int64_t g = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (g >= total_frames) return;
  if (WIN) {
    int seg; int64_t k;
    if (!row_in_window(win, g, seg, k)) {
      if (lane == 0) row_count[g] = 0;
      return;
    }
  }
  const uint32_t *row = bitmap + g * kBitmapRowWords;
  int c = 0;
  if (STRIPED) {
    if (lane < kW2Strips) {
      const uint4 w = *reinterpret_cast<const uint4 *>(row + 4 * lane);
      c = __popc(w.x) + __popc(w.y) + __popc(w.z) + __popc(w.w);
    }
  } else {
    c = __popc(row[lane]) + __popc(row[lane + 32]);
    if (lane == 0) c += __popc(row[64]);
  }
#pragma unroll
  for (int d = 16; d; d >>= 1) c += __shfl_xor_sync(0xffffffffu, c, d);
  if (lane == 0) row_count[g] = (uint32_t)c;
}

template <bool STRIPED, bool WIN>
__global__ void __launch_bounds__(256)
extract_kernel(const uint32_t *__restrict__ bitmap, const int64_t *__restrict__ row_off,
               const int64_t *__restrict__ frame_starts, int n_tracks, int64_t total_frames, int64_t peak_base,
               int32_t *__restrict__ peak_t, int32_t *__restrict__ peak_f, int64_t cap,
               int64_t *__restrict__ track_peak_starts, int32_t *__restrict__ status, const PeakWindow win) {
  const int lane = threadIdx.x & 31;
  const int64_t g = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (g >= total_frames) return;
  int trk;
  int k;
  int64_t base = row_off[g] + peak_base;
  if (WIN) {
    int64_t kl;
    if (!row_in_window(win, g, trk, kl)) return;
    k = (int)(kl + win.t_base[trk]);
    base += win.peak_off[trk];
  } else {
    trk = find_segment(frame_starts, n_tracks, g);
    k = (int)(g - frame_starts[trk]);
  }
  if (!WIN && lane == 0) {
    // prefix offsets never point past the workspace: the peaks beyond `cap` are dropped (status bit 1), and the
    // kernels that follow (pair counting, scans, SHA-1) read these counts from the device
    if (k == 0) track_peak_starts[trk] = min(base, cap);
    if (g == total_frames - 1) track_peak_starts[n_tracks] = min(row_off[total_frames] + peak_base, cap);
  }
  const uint32_t *row = bitmap + g * kBitmapRowWords;
  bool overflow = false;
  auto excl_scan = [&](int cnt, int &total) {
    int incl = cnt;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      int o = __shfl_up_sync(0xffffffffu, incl, d);
      if (lane >= d) incl += o;
    }
    total = __shfl_sync(0xffffffffu, incl, 31);
    return incl - cnt;
  };
  if (STRIPED) {
    uint4 w = make_uint4(0, 0, 0, 0);
    if (lane < kW2Strips) w = *reinterpret_cast<const uint4 *>(row + 4 * lane);
    const int cnt = __popc(w.x) + __popc(w.y) + __popc(w.z) + __popc(w.w);
    int total;
    int64_t idx = base + excl_scan(cnt, total);
    uint32_t any = w.x | w.y | w.z | w.w;
    while (any) {                                   // ascending bin order: lane-bit l major, element e minor
      const int l = __ffs(any) - 1;
      any &= any - 1;
      const uint32_t nib = ((w.x >> l) & 1u) | (((w.y >> l) & 1u) << 1) | (((w.z >> l) & 1u) << 2) | (((w.w >> l) & 1u) << 3);
#pragma unroll
      for (int e = 0; e < 4; ++e)
        if ((nib >> e) & 1u) {
          if (idx < cap) { peak_t[idx] = k; peak_f[idx] = kW2Bins * lane + 4 * l + e; } else overflow = true;
          ++idx;
        }
    }
  } else {
#pragma unroll
    for (int round = 0; round < 3; ++round) {
      const int w = round * 32 + lane;
      uint32_t word = w < SIA_ROW_WORDS ? row[w] : 0u;
      const int cnt = __popc(word);
      int total;
      int64_t idx = base + excl_scan(cnt, total);
      while (word) {
        const int bit = __ffs(word) - 1;
        word &= word - 1;
        if (idx < cap) { peak_t[idx] = k; peak_f[idx] = w * 32 + bit; } else overflow = true;
        ++idx;
      }
      base += total;
    }
  }
  if (overflow) atomicOr(status, 1);
}

}  // namespace

int peaks_bitmap_launch(const PeaksLaunch &a, cudaStream_t s, bool *striped) {
  *striped = false;
  if (a.total_ttiles == 0) return SIA_OK;
  SIA_REQUIRE(a.nbhd >= 1 && a.nbhd <= SIA_MAX_NBHD, SIA_E_UNSUPPORTED, "peaks: nbhd must be in 1..64");
  SIA_REQUIRE(a.connectivity == 1 || a.connectivity == 2, SIA_E_UNSUPPORTED, "peaks: connectivity must be 1 or 2");
  const bool erosion = a.amp_min < 0;
  if (a.connectivity == 2 && a.nbhd == 10) {
    // (double + erosion would need 255 KB of shared memory: it takes the footprint kernel)
    if (a.in_type == SIA_F64 && !erosion) return launch_square<double, 10, false>(a, s);
    if (a.in_type == SIA_F32 && !erosion) {
      *striped = true;
      return launch_square_warp(a, s);
    }
    if (a.in_type == SIA_F32) return launch_square<float, 10, true>(a, s);
  }
  if (a.connectivity == 1 && a.nbhd <= brute_max_nbhd(a.in_type))
    return a.in_type == SIA_F64 ? launch_generic<double>(a, s) : launch_generic<float>(a, s);
  if (a.in_type == SIA_F64) return erosion ? launch_footprint<double, true>(a, s) : launch_footprint<double, false>(a, s);
  return erosion ? launch_footprint<float, true>(a, s) : launch_footprint<float, false>(a, s);
}

int peaks_rowcount_launch(const uint32_t *d_bitmap, bool striped, int64_t total_frames, uint32_t *d_row_count,
                          cudaStream_t s, const PeakWindow *win) {
  if (total_frames == 0) return SIA_OK;
  const unsigned blocks = (unsigned)ceil_div(total_frames * 32, 256);
  const PeakWindow w = win ? *win : PeakWindow{};
  if (win) {
    if (striped) rowcount_kernel<true, true><<<blocks, 256, 0, s>>>(d_bitmap, total_frames, d_row_count, w);
    else rowcount_kernel<false, true><<<blocks, 256, 0, s>>>(d_bitmap, total_frames, d_row_count, w);
  } else {
    if (striped) rowcount_kernel<true, false><<<blocks, 256, 0, s>>>(d_bitmap, total_frames, d_row_count, w);
    else rowcount_kernel<false, false><<<blocks, 256, 0, s>>>(d_bitmap, total_frames, d_row_count, w);
  }
  SIA_CHECK_LAUNCH();
  return SIA_OK;
}

int peaks_extract_launch(const uint32_t *d_bitmap, bool striped, const int64_t *d_row_off,
                         const int64_t *d_frame_starts, int n_tracks, int64_t total_frames, int64_t peak_base, int32_t *d_peak_t,
                         int32_t *d_peak_f, int64_t cap_peaks, int64_t *d_track_peak_starts, int32_t *d_status,
                         cudaStream_t s, const PeakWindow *win) {
  if (total_frames == 0) return SIA_OK;
  const unsigned blocks = (unsigned)ceil_div(total_frames * 32, 256);
  const PeakWindow w = win ? *win : PeakWindow{};
#define SIA_EXTRACT(ST, WN)                                                                                       \
  extract_kernel<ST, WN><<<blocks, 256, 0, s>>>(d_bitmap, d_row_off, d_frame_starts, n_tracks, total_frames, peak_base, \
                                                d_peak_t, d_peak_f, cap_peaks, d_track_peak_starts, d_status, w)
  if (win) {
    if (striped) SIA_EXTRACT(true, true); else SIA_EXTRACT(false, true);
  } else {
    if (striped) SIA_EXTRACT(true, false); else SIA_EXTRACT(false, false);
  }
#undef SIA_EXTRACT
  SIA_CHECK_LAUNCH();
  return SIA_OK;
}

}  // namespace sia
