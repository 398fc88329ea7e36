// K1 — batched 4096-point STFT -> dB spectrogram, replacing
//   mlab.specgram(x, NFFT=4096, Fs, window_hanning, noverlap=2048)[0]   (__init__.py:232-237)
//   (any noverlap 0..4095 through the kAnyHop staging below; 2048 = wratio 0.5 is the tuned path)
//   10*log10(P) with P==0 -> 0                                           (__init__.py:241)
//
// One CTA (128 threads) transforms one frame at a time and walks a run of consecutive
// frames.  The real 4096-point FFT is done as a 2048-point complex FFT of the
// even/odd-packed windowed samples plus a split post-pass; the complex FFT is three
// register passes (radix 16, 16, 8) through shared memory:
//
//   n = 128a + 8b + c      k = ka + 16kb + 256kc
//   pass A  thread t=8b+c   : FFT16 over a, x W2048^(t*ka)      -> L1[ka*136 + t]
//   pass B  thread (ka,c)   : FFT16 over b, x W128^(c*kb)       -> L2[c*258 + kb*16 + ka]
//   pass C  thread t: FFT8 over c of columns u = t and 256-t (u = kb*16+ka)  -> Z[u + 256kc] in registers
//   post    the same thread holds Z[k] and Z[2048-k]: E +/- W4096^k O, |.|^2, dB -> global, coalesced
//
// The strides 136 and 258 make every shared-memory access of every pass conflict-free
// for 8-byte (and 4-byte) elements.  PCM is read straight from global memory as packed
// int16 pairs (each warp load is one 128-byte line; the 50% overlap re-read hits L2).
//
// T = double is the default arithmetic: with 144 dB between the strongest and weakest
// bins of a frame, float butterflies leave O(1) relative error on the weak bins, which
// breaks the 1e-3 dB bound against the reference's float64 spectrogram.  T = float is
// kept as a selectable fast mode.
#include "sia_common.cuh"
#include "stft.cuh"

#include <cstdlib>
#include <math.h>
#include <vector>

namespace sia {

namespace {

template <typename T> struct Vec2;
template <> struct Vec2<float> { using type = float2; };
template <> struct Vec2<double> { using type = double2; };

#ifndef SIA_STFT_CTAS_F64
#define SIA_STFT_CTAS_F64 4
#endif
constexpr int kStftCtasF64 = SIA_STFT_CTAS_F64;   // resident CTAs per SM of the float64 kernel (5 fit in shared memory and 96 registers, measured no faster: the FP64 pipe is the limit)
constexpr int kL1Stride = 136;
// pass-C layout stride in (re, im) elements: odd for 16-byte elements (a quarter-warp of 8 lanes stores c = 0..7 at one
// ka), 2 mod 16 for 8-byte elements (a half-warp stores c = 0..7 at two consecutive ka)
constexpr int kBufElems = 16 * kL1Stride;  // 2176 >= 8*258=2064 >= 2048

template <typename T>
__device__ __forceinline__ void cmul(T &r, T &i, T wr, T wi) {
  T nr = r * wr - i * wi;
  T ni = r * wi + i * wr;
  r = nr; i = ni;
}

template <typename T>
__device__ __forceinline__ void fft4(T &r0, T &i0, T &r1, T &i1, T &r2, T &i2, T &r3, T &i3) {
  T ar = r0 + r2, ai = i0 + i2;
  T br = r0 - r2, bi = i0 - i2;
  T cr = r1 + r3, ci = i1 + i3;
  T dr = r1 - r3, di = i1 - i3;
  r0 = ar + cr; i0 = ai + ci;
  r2 = ar - cr; i2 = ai - ci;
  r1 = br + di; i1 = bi - dr;   // b - i*d
  r3 = br - di; i3 = bi + dr;   // b + i*d
}

// In-place 16-point forward FFT.  Output X[k], k = k1 + 4*k2, lands at position 4*k1 + k2.
template <typename T>
__device__ __forceinline__ void fft16(T (&r)[16], T (&i)[16]) {
  const T C1 = (T)0.92387953251128675613;   // cos(pi/8)
  const T S1 = (T)0.38268343236508977173;   // sin(pi/8)
  const T H = (T)0.70710678118654752440;    // sqrt(1/2)
#pragma unroll
  for (int n2 = 0; n2 < 4; ++n2)
    fft4(r[n2], i[n2], r[n2 + 4], i[n2 + 4], r[n2 + 8], i[n2 + 8], r[n2 + 12], i[n2 + 12]);
  // element (n2 + 4*k1) *= W16^(n2*k1),  W16^m = (cos(m pi/8), -sin(m pi/8))
  cmul(r[5], i[5], C1, -S1);                                  // m=1
  { T a = r[6], b = i[6]; r[6] = (a + b) * H; i[6] = (b - a) * H; }   // m=2: (1-i)/sqrt2
  cmul(r[7], i[7], S1, -C1);                                  // m=3
  { T a = r[9], b = i[9]; r[9] = (a + b) * H; i[9] = (b - a) * H; }   // m=2
  { T a = r[10], b = i[10]; r[10] = b; i[10] = -a; }          // m=4: -i
  { T a = r[11], b = i[11]; r[11] = (b - a) * H; i[11] = -(a + b) * H; }  // m=6: (-1-i)/sqrt2
  cmul(r[13], i[13], S1, -C1);                                // m=3
  { T a = r[14], b = i[14]; r[14] = (b - a) * H; i[14] = -(a + b) * H; }  // m=6
  cmul(r[15], i[15], -C1, S1);                                // m=9 = -W^1
#pragma unroll
  for (int k1 = 0; k1 < 4; ++k1)
    fft4(r[4 * k1], i[4 * k1], r[4 * k1 + 1], i[4 * k1 + 1], r[4 * k1 + 2], i[4 * k1 + 2], r[4 * k1 + 3],
         i[4 * k1 + 3]);
}
__host__ __device__ constexpr int pos16(int k) { return 4 * (k & 3) + (k >> 2); }

// In-place 8-point forward FFT.  Output X[k], k = k1 + 4*k2, lands at position 2*k1 + k2.
template <typename T>
__device__ __forceinline__ void fft8(T (&r)[8], T (&i)[8]) {
  const T H = (T)0.70710678118654752440;
#pragma unroll
  for (int n2 = 0; n2 < 2; ++n2)
    fft4(r[n2], i[n2], r[n2 + 2], i[n2 + 2], r[n2 + 4], i[n2 + 4], r[n2 + 6], i[n2 + 6]);
  // element (1 + 2*k1) *= W8^k1
  { T a = r[3], b = i[3]; r[3] = (a + b) * H; i[3] = (b - a) * H; }       // k1=1
  { T a = r[5], b = i[5]; r[5] = b; i[5] = -a; }                          // k1=2: -i
  { T a = r[7], b = i[7]; r[7] = (b - a) * H; i[7] = -(a + b) * H; }      // k1=3
#pragma unroll
  for (int k1 = 0; k1 < 4; ++k1) {
    T ar = r[2 * k1], ai = i[2 * k1], br = r[2 * k1 + 1], bi = i[2 * k1 + 1];
    r[2 * k1] = ar + br; i[2 * k1] = ai + bi;
    r[2 * k1 + 1] = ar - br; i[2 * k1 + 1] = ai - bi;
  }
}
__host__ __device__ constexpr int pos8(int k) { return 2 * (k & 3) + (k >> 2); }

// ---- constants in the constant bank (operands of DFMA/FFMA, no load instruction) ----------------------
__constant__ double2 c_winA_d[16];   // (cos, sin)(2*pi*256*a/4095)
__constant__ float2 c_winA_f[16];
__constant__ double2 c_w32_d[8];     // W32^it = (cos, -sin)(2*pi*it/32)
__constant__ float2 c_w32_f[8];
__constant__ double2 c_spc_d[9];     // W4096^k of the self-mirrored columns: k = 256 i (i<5), 128 + 256 (i-5)
__constant__ float2 c_spc_f[9];
template <typename T> __device__ __forceinline__ typename Vec2<T>::type spc_tw(int i);
template <> __device__ __forceinline__ double2 spc_tw<double>(int i) { return c_spc_d[i]; }
template <> __device__ __forceinline__ float2 spc_tw<float>(int i) { return c_spc_f[i]; }
template <typename T> __device__ __forceinline__ typename Vec2<T>::type winA(int a);
template <> __device__ __forceinline__ double2 winA<double>(int a) { return c_winA_d[a]; }
template <> __device__ __forceinline__ float2 winA<float>(int a) { return c_winA_f[a]; }
template <typename T> __device__ __forceinline__ typename Vec2<T>::type w32(int k);
template <> __device__ __forceinline__ double2 w32<double>(int k) { return c_w32_d[k]; }
template <> __device__ __forceinline__ float2 w32<float>(int k) { return c_w32_f[k]; }

// int16 sample -> real, exactly.  float64: one I2F.F64.S32 per sample (conversion pipe); the alternative
// (-DSIA_STFT_SPLICE, and the float32 kernel) splices the integer into the mantissa of 2^52+2^31 (resp. 1.5*2^23) and
// subtracts the magic constant on the FP pipe.
template <typename T> __device__ __forceinline__ T sample_to_real(int s);
template <> __device__ __forceinline__ double sample_to_real<double>(int s) {
#ifndef SIA_STFT_SPLICE
  return (double)s;                     // I2F.F64.S32: runs on the conversion pipe, beside the FP64 / integer pipes K1 is
                                        // bound by (38.2 -> 37.5 ms per 1000 tracks against the mantissa splice below)
#else
  return __hiloint2double(0x43300000, (int)(0x80000000u ^ (uint32_t)s)) - 4503601774854144.0;
#endif
}
template <> __device__ __forceinline__ float sample_to_real<float>(int s) {
  return __int_as_float(0x4b400000 + s) - 12582912.0f;
}
// the two int16 samples of a packed PCM word.  float64: converting from `short` lets the compiler read the halves of
// the register directly (I2F.F64.S16 R, R / R.H1): no extraction instruction on the integer pipe
template <typename T> __device__ __forceinline__ void sample_pair(uint32_t w, T &s0, T &s1) {
  s0 = sample_to_real<T>((int)(short)(w & 0xffffu));
  s1 = sample_to_real<T>((int)w >> 16);
}
#ifndef SIA_STFT_SPLICE
template <> __device__ __forceinline__ void sample_pair<double>(uint32_t w, double &s0, double &s1) {
  s0 = (double)(short)(w & 0xffffu);
  s1 = (double)(short)(w >> 16);
}
#endif

// dB epilogue.  dB = 10*log10(p*scale) = C*(e + Ki + log2(m) + Kf),  C = 10*log10(2), p = m*2^e, log2(scale) = Ki+Kf.
// p is rounded to float once (F2F), log2 of its mantissa is one MUFU.LG2 (absolute error ~2^-22); the integer part
// is recombined with a split constant (E*C_hi is exact), so the result carries 0.5 ulp(float) + ~1.4e-6 dB.
// p == 0 -> 0 dB (__init__.py:241).  Branch-free.
struct DbScale { int ke; float kf; double c; float kif; };     // ke = Ki - 1023, kif = (float)Ki
constexpr float kC = 3.01029995663981195f;
constexpr float kC_hi = 6165.0f / 2048.0f;                                   // 13 significant bits
constexpr float kC_lo = (float)(3.01029995663981195 - 6165.0 / 2048.0);

// MUFU.LG2 alone: __log2f wraps it in a denormal rescue (FSETP + FMUL + FADD) that the inputs here never need
__device__ __forceinline__ float lg2_raw(float x) {
  float y;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

__device__ __forceinline__ float db_combine(int E, float L) {
  const float Ef = __int_as_float(0x4b400000 + E) - 12582912.0f;             // exact int -> float, |E| < 2^22
  return fmaf(Ef, kC_hi, fmaf(Ef, kC_lo, L * kC));
}
template <typename OutT>
__device__ __forceinline__ OutT db_out(double p, const DbScale &sc) {
  if (sizeof(OutT) == 8)                                                     // float64 output (tests): exact path
    return (OutT)(p == 0.0 ? 0.0 : 10.0 * log10(p) + sc.c);
  // one conversion (round to nearest: the 24-bit mantissa the logarithm sees), then the float's exponent and
  // mantissa fields; |X|^2 of int16 PCM lies in [1e-26, 1e21], inside the float range
  const float pf = __double2float_rn(p);
  const int b = __float_as_int(pf);
  // exponent and mantissa each through MUFU.LG2 (log2 of a power of two is exact): two mask instructions are all the
  // integer pipe sees — K1 is bound by FP64 + integer pipe time, the MUFU pipe is idle
  const float Ef = lg2_raw(__int_as_float(b & 0x7f800000)) + sc.kif;
  const float L = lg2_raw(__int_as_float((b & 0x007fffff) | 0x3f800000)) + sc.kf;
  const float r = fmaf(Ef, kC_hi, fmaf(Ef, kC_lo, L * kC));
  return (OutT)(pf == 0.f ? 0.f : r);
}
template <typename OutT>
__device__ __forceinline__ OutT db_out(float p, const DbScale &sc) {
  const int b = max(__float_as_int(p), 0x00800000);                          // clamp float subnormals
  const float r = db_combine((b >> 23) - 127 + sc.ke + 1023,
                             __log2f(__int_as_float((b & 0x7fffff) | 0x3f800000)) + sc.kf);
  return (OutT)(p == 0.f ? 0.f : r);
}

// bins k and 2048-k from A = Z[k], B = Z[2048-k], tw = W4096^k (split post-pass of the packed real FFT)
template <typename T, typename OutT>
__device__ __forceinline__ void emit_pair(OutT *__restrict__ row, T ar, T ai, T br, T bi, T twr, T twi, int k,
                                          const DbScale &sc) {
  const T er = ar + br, ei = ai - bi;                // 2E = A + conj(B)
  const T orr = ai + bi, oi = br - ar;               // 2O = -i (A - conj(B))
  const T tr = orr * twr - oi * twi, ti = orr * twi + oi * twr;
  const T pr = er + tr, pi = ei + ti;                // 2 X[k]
  const T qr = er - tr, qi = ei - ti;                // 2 conj(X[2048-k])
  row[k] = db_out<OutT>(pr * pr + pi * pi, sc);
  row[2048 - k] = db_out<OutT>(qr * qr + qi * qi, sc);
}

// the 17 bins of the self-mirrored columns 0 and 128 (parked by thread 0), one pair per lane i = 0..8
template <typename T, typename OutT>
__device__ __forceinline__ void emit_special(OutT *__restrict__ row, const T *__restrict__ pr, const T *__restrict__ pi,
                                             int i, const DbScale &sc_mid, const DbScale &sc_edge) {
  const int a = i < 5 ? i : 8 + (i - 5);              // A index: column 0 kc = i, or column 128 kc = i-5
  const int b = i < 5 ? ((8 - i) & 7) : 8 + (12 - i); // its mirror in the same column
  const int k = i < 5 ? 256 * i : 128 + 256 * (i - 5);
  const typename Vec2<T>::type tw = spc_tw<T>(i);
  emit_pair<T, OutT>(row, pr[a], pi[a], pr[b], pi[b], tw.x, tw.y, k, k == 0 ? sc_edge : sc_mid);
}

// PCM ring of the any-hop staging (kAnyHop): 513 16-byte chunks = 4104 samples, one chunk more than a frame, because
// a frame that starts off an 8-sample boundary touches 513 chunks.  Chunk c of a track (samples [8c, 8c+8)) lives in
// slot c mod 513, so sample n of the track is ring word (n/2) mod 2052.  Word 2052 mirrors word 0, so the word after
// any ring word is read without a wrap test.
constexpr int kRingChunks = 513;
constexpr int kRingSamples = 8 * kRingChunks;
constexpr int kRingWords = kRingSamples / 2;

// kAnyHop = false: frame k of a track starts at sample 2048 k (wratio 0.5), staged in two half-blocks.
// kAnyHop = true:  frame k starts at sample k * hop, hop in 1..4096, staged in the 513-chunk ring above.
// Passes A-C and the dB epilogue are shared: a frame gives the same bits whatever the hop.
template <typename T, typename OutT, bool kAnyHop>
__global__ void __launch_bounds__(128, sizeof(T) == 8 ? kStftCtasF64 : 6)
stft_db_kernel(const int16_t *__restrict__ pcm, const int64_t *__restrict__ track_starts,
               const int64_t *__restrict__ track_len, const int64_t *__restrict__ frame_starts, int n_tracks,
               int64_t total_frames, int frames_per_cta, OutT *__restrict__ out, DbScale sc_mid, DbScale sc_edge,
               const typename Vec2<T>::type *__restrict__ winB, const typename Vec2<T>::type *__restrict__ twA,
               const typename Vec2<T>::type *__restrict__ twB, const typename Vec2<T>::type *__restrict__ twP, int hop) {
  using V2 = typename Vec2<T>::type;
  __shared__ __align__(16) V2 sbuf[kBufElems];      // (re, im) interleaved: one 128-bit (64-bit) access per element
  constexpr int kL2Stride = sizeof(T) == 8 ? 257 : 258;

  // PCM ring: two 2048-sample half-blocks.  Frame k of a track reads half-blocks k and k+1 (slots k&1, ~k&1) in
  // pass A; once pass A is over (first barrier) the half-block the NEXT frame adds, k+2, is fetched with
  // cp.async into the slot of half-block k while passes B and C run, so the DRAM latency of the PCM never sits
  // in front of pass A.  Bytes past the end of a track are zero-filled (src-size), which is exactly
  // mlab.specgram's zero padding of a short input.
  // kAnyHop: the same schedule on the 513-chunk ring (kRingWords + 1 words used): after pass A of frame k, the
  // chunks frame k+1 adds are fetched into the slots of chunks no later frame reads.
  __shared__ __align__(16) uint32_t spcm[2][kAnyHop ? 1028 : 1024];
  __shared__ T sspc[2][2][16];     // parked columns 0 / 128 of the last two frames (re, im)

  const int t = threadIdx.x;

  int64_t g = (int64_t)blockIdx.x * frames_per_cta;
  if (g >= total_frames) return;
  int64_t g_end = g + frames_per_cta;
  if (g_end > total_frames) g_end = total_frames;
  int trk = find_segment(frame_starts, n_tracks, g);

  const uint32_t spcm_base = (uint32_t)__cvta_generic_to_shared(&spcm[0][0]);
  // PCM cursor: this thread's first 16-byte chunk of the next half-block to stage and the bytes of the track left from
  // there, clamped to +-2^30 (set at the start of every run / track, a run is a few frames: the clamp never bites)
  const char *cur_src = nullptr;
  int cur_rest = 0;
  auto set_cursor = [&](int tr, int64_t h) {
    const int64_t rest = (track_len[tr] - h * SIA_HOP) * 2 - 16 * t;
    cur_rest = (int)max(min(rest, (int64_t)1 << 30), -((int64_t)1 << 30));
    cur_src = reinterpret_cast<const char *>(pcm + track_starts[tr] + h * SIA_HOP) + 16 * t;
  };
  auto fetch_half = [&](int slot) {
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int nbytes = min(max(cur_rest - 2048 * i, 0), 16);
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(spcm_base + (uint32_t)(slot * 4096 + 16 * t + 2048 * i)),
                   "l"(nbytes ? cur_src + 2048 * i : reinterpret_cast<const char *>(pcm)), "r"(nbytes));
    }
    cur_src += 2 * SIA_HOP;
    cur_rest -= 2 * SIA_HOP;
  };
  int slot = 0;
  bool primed = false;

  // kAnyHop: the ring holds the track's samples up to fe, a multiple of 8; cur_src / cur_rest are the track's PCM and
  // bytes left from fe on.  For the current frame, starting at sample s: s_mod = s mod kRingSamples, lead = fe - s
  // (-7..4103).  kRingSamples is a multiple of 8, so s and s_mod share their residue mod 8.
  int s_mod = 0, lead = 0;
  auto set_ring = [&](int tr, int64_t k) {
    const int64_t s = k * hop, fe = s & ~(int64_t)7;
    s_mod = (int)(s % kRingSamples);
    lead = (int)(fe - s);
    const int64_t rest = (track_len[tr] - fe) * 2;
    cur_rest = (int)max(min(rest, (int64_t)1 << 30), -((int64_t)1 << 30));
    cur_src = reinterpret_cast<const char *>(pcm + track_starts[tr] + fe);
  };
  auto fetch_frame = [&]() {      // the chunks from fe up to the end of the current frame: at most kRingChunks
    const int n = (SIA_NFFT - lead + 7) >> 3;
    int fe_mod = s_mod + lead;
    if (fe_mod < 0) fe_mod += kRingSamples;
    if (fe_mod >= kRingSamples) fe_mod -= kRingSamples;
    for (int i = t; i < n; i += 128) {
      int pos = fe_mod + 8 * i;
      if (pos >= kRingSamples) pos -= kRingSamples;
      const int nbytes = min(max(cur_rest - 16 * i, 0), 16);
      const char *src = nbytes ? cur_src + 16 * i : reinterpret_cast<const char *>(pcm);
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(spcm_base + 2 * (uint32_t)pos), "l"(src),
                   "r"(nbytes));
      if (pos == 0)      // the mirror word behind the ring
        asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;\n" ::"r"(spcm_base + 4 * (uint32_t)kRingWords),
                     "l"(src), "r"(min(nbytes, 4)));
    }
    lead += 8 * n;
    cur_src += 16 * n;
    cur_rest -= 16 * n;
  };
  auto next_frame = [&]() {
    s_mod += hop;
    if (s_mod >= kRingSamples) s_mod -= kRingSamples;
    lead -= hop;
  };

  const int64_t g_first = g;
  for (; g < g_end; ++g) {
    // lanes 1..9: finish the previous frame (its parked columns became visible at the barrier)
    if (g > g_first && t >= 1 && t <= 9)
      emit_special<T, OutT>(out + (g - 1) * (int64_t)SIA_F_STRIDE, sspc[(g - 1) & 1][0], sspc[(g - 1) & 1][1], t - 1,
                            sc_mid, sc_edge);
    while (g >= frame_starts[trk + 1]) ++trk;
    const int64_t k = g - frame_starts[trk];
    if (!primed) {                       // first frame of the run or of a track: both half-blocks, synchronously
      if constexpr (kAnyHop) {
        set_ring(trk, k);
        fetch_frame();
      } else {
        set_cursor(trk, k);
        fetch_half(slot);
        fetch_half(slot ^ 1);
      }
      asm volatile("cp.async.wait_all;\n" ::: "memory");
      __syncthreads();
    }
    primed = g + 1 < frame_starts[trk + 1];           // the next frame continues this track

    T xr[16], xi[16];
    // ---- pass A: window, pack even/odd samples as complex, FFT16 over a -----------------
    {
      uint32_t w[16];
      if constexpr (kAnyHop) {
        // samples s + 256a + 2t, +1: ring words j, j+1 shifted right by 16 bits when s is odd
        const uint32_t *__restrict__ ring = &spcm[0][0];
        const int sh = (s_mod & 1) << 4;
        int j = (s_mod >> 1) + t;
        if (j >= kRingWords) j -= kRingWords;
#pragma unroll
        for (int a = 0; a < 16; ++a) {
          w[a] = __funnelshift_r(ring[j], ring[j + 1], sh);
          j += 128;
          if (j >= kRingWords) j -= kRingWords;
        }
      } else {
        const uint32_t *__restrict__ h0 = spcm[slot], *__restrict__ h1 = spcm[slot ^ 1];
#pragma unroll
        for (int a = 0; a < 8; ++a) { w[a] = h0[128 * a + t]; w[a + 8] = h1[128 * a + t]; }
      }
      const V2 wb0 = __ldg(winB + 2 * t), wb1 = __ldg(winB + 2 * t + 1);   // window phase of samples 2t, 2t+1
      // np.hanning: w[m] = 0.5 - 0.5*cos(2*pi*m/4095), m = 256a + 2t (+1).  cos(a*D + B_t), D = 2*pi*256/4095, by the
      // three-term recurrence c[a+1] = 2cos(D) c[a] - c[a-1]: one FMA per sample (16 steps: error growth ~1e-15)
      const V2 cd = winA<T>(1);
      const T K2 = cd.x + cd.x;
      T c0p = wb0.x, c1p = wb1.x;                                   // c[a-1]
      T c0 = cd.x * wb0.x - cd.y * wb0.y, c1 = cd.x * wb1.x - cd.y * wb1.y;   // c[a], a = 1
#pragma unroll
      for (int a = 0; a < 16; ++a) {
        T ca0, ca1;
        if (a == 0) { ca0 = c0p; ca1 = c1p; }
        else if (a == 1) { ca0 = c0; ca1 = c1; }
        else {
          ca0 = fma(K2, c0, -c0p); ca1 = fma(K2, c1, -c1p);
          c0p = c0; c1p = c1; c0 = ca0; c1 = ca1;
        }
        // x*(1 - cos) = 2*x*w: one FMA; the factor 2 is folded into the dB constant
        T s0, s1;
        sample_pair<T>(w[a], s0, s1);
        xr[a] = fma(-s0, ca0, s0);
        xi[a] = fma(-s1, ca1, s1);
      }
      fft16(xr, xi);
      // twiddles W2048^(t*ka): four loaded (ka = 1, 2, 4, 8), the rest by products (<= 3 deep)
      const V2 b1 = __ldg(twA + 1 * 128 + t), b2 = __ldg(twA + 2 * 128 + t);
      const V2 b4 = __ldg(twA + 4 * 128 + t), b8 = __ldg(twA + 8 * 128 + t);
      auto put = [&](int ka, T wr, T wi) {
        T r = xr[pos16(ka)], i = xi[pos16(ka)];
        cmul(r, i, wr, wi);
        V2 o; o.x = r; o.y = i;
        sbuf[ka * kL1Stride + t] = o;
      };
      auto mul = [](V2 a, V2 b) { V2 o; o.x = a.x * b.x - a.y * b.y; o.y = a.x * b.y + a.y * b.x; return o; };
      { V2 o; o.x = xr[0]; o.y = xi[0]; sbuf[t] = o; }
#ifdef SIA_STFT_TWA_ALL
      put(1, b1.x, b1.y); put(2, b2.x, b2.y); put(4, b4.x, b4.y); put(8, b8.x, b8.y);
#pragma unroll
      for (int ka = 3; ka < 16; ++ka)
        if (ka & (ka - 1)) { const V2 w = __ldg(twA + ka * 128 + t); put(ka, w.x, w.y); }    // all 15 from the table
#else
      put(1, b1.x, b1.y); put(2, b2.x, b2.y);
      { const V2 w3 = mul(b2, b1); put(3, w3.x, w3.y); }
      put(4, b4.x, b4.y);
      { const V2 w5 = mul(b4, b1); put(5, w5.x, w5.y); }
      { const V2 w6 = mul(b4, b2); put(6, w6.x, w6.y); const V2 w7 = mul(w6, b1); put(7, w7.x, w7.y); }
      put(8, b8.x, b8.y);
      { const V2 w9 = mul(b8, b1); put(9, w9.x, w9.y); }
      { const V2 w10 = mul(b8, b2); put(10, w10.x, w10.y); const V2 w11 = mul(w10, b1); put(11, w11.x, w11.y); }
      { const V2 w12 = mul(b8, b4); put(12, w12.x, w12.y);
        const V2 w13 = mul(w12, b1); put(13, w13.x, w13.y);
        const V2 w14 = mul(w12, b2); put(14, w14.x, w14.y);
        const V2 w15 = mul(w14, b1); put(15, w15.x, w15.y); }
#endif
    }
    __syncthreads();
    if (primed && g + 1 < g_end) {
      if constexpr (kAnyHop) { next_frame(); fetch_frame(); }     // what frame k+1 adds; pass A is done with frame k
      else fetch_half(slot);                                       // half-block k+2; pass A has consumed this slot
    }
    // ---- pass B: FFT16 over b -----------------------------------------------------------
    {
      const int ka = t >> 3, c = t & 7;
#pragma unroll
      for (int b = 0; b < 16; ++b) {
        const V2 v = sbuf[ka * kL1Stride + 8 * b + c];
        xr[b] = v.x; xi[b] = v.y;
      }
      __syncthreads();
      fft16(xr, xi);
#pragma unroll
      for (int kb = 0; kb < 16; ++kb) {
        T r = xr[pos16(kb)], i = xi[pos16(kb)];
        if (kb) {
          const V2 tw = __ldg(twB + kb * 8 + c);
          cmul(r, i, tw.x, tw.y);
        }
        V2 o; o.x = r; o.y = i;
        sbuf[c * kL2Stride + kb * 16 + ka] = o;
      }
    }
    __syncthreads();
    // ---- pass C + split post-pass, fused in registers ---------------------------------------------
    // Z[k] and its mirror Z[2048-k] are produced by columns u and 256-u of pass C (k = u + 256kc,
    // 2048-k = (256-u) + 256(7-kc)), so thread t takes columns t and 256-t and never writes Z back to
    // shared memory.  Thread 0 takes the two self-mirrored columns 0 and 128 (17 bins instead of 16).
    {
      T yr[2][8], yi[2][8];
      const int u1 = t == 0 ? 128 : 256 - t;
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        const V2 v0 = sbuf[c * kL2Stride + t], v1 = sbuf[c * kL2Stride + u1];
        yr[0][c] = v0.x; yi[0][c] = v0.y;
        yr[1][c] = v1.x; yi[1][c] = v1.y;
      }
      fft8(yr[0], yi[0]);
      fft8(yr[1], yi[1]);
      if (t == 0) {
        // columns 0 and 128 mirror onto themselves: park them; nine lanes emit their 17 bins after the barrier
        T *pr = sspc[g & 1][0], *pi = sspc[g & 1][1];
#pragma unroll
        for (int kc = 0; kc < 8; ++kc) {
          pr[kc] = yr[0][pos8(kc)]; pi[kc] = yi[0][pos8(kc)];
          pr[8 + kc] = yr[1][pos8(kc)]; pi[8 + kc] = yi[1][pos8(kc)];
        }
      } else {
        OutT *__restrict__ row = out + g * (int64_t)SIA_F_STRIDE;
        // W4096^(t + 256 j): j = 0..3 from the table (k <= 895), j = 4..7 by W^(k + 1024) = -i W^k — four loads,
        // no products (K1 is bound by FP64 + integer pipe time, the load pipe has room)
        V2 twj[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) twj[j] = __ldg(twP + t + 256 * j);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const T wr = j < 4 ? twj[j].x : twj[j - 4].y;
          const T wi = j < 4 ? twj[j].y : -twj[j - 4].x;
          emit_pair<T, OutT>(row, yr[0][pos8(j)], yi[0][pos8(j)], yr[1][pos8(7 - j)], yi[1][pos8(7 - j)], wr, wi,
                             t + 256 * j, sc_mid);
        }
      }
    }
    asm volatile("cp.async.wait_all;\n" ::: "memory");   // next frame's half-block has landed
    __syncthreads();   // ... and the L2 layout may be overwritten by the next frame's pass A
    slot ^= 1;
  }
  if (t >= 1 && t <= 9)
    emit_special<T, OutT>(out + (g_end - 1) * (int64_t)SIA_F_STRIDE, sspc[(g_end - 1) & 1][0], sspc[(g_end - 1) & 1][1],
                          t - 1, sc_mid, sc_edge);
}

}  // namespace

// ---------------------------------------------------------------------------------------------
// tables
// ---------------------------------------------------------------------------------------------
template <typename T>
static int upload_tables(StftTables<T> &tb) {
  using V2 = typename Vec2<T>::type;
  const long double PI = 3.141592653589793238462643383279502884L;
  std::vector<V2> win(256), twA(16 * 128), twB(16 * 8), twP(1025);
  for (int m = 0; m < 256; ++m) {
    // np.hanning(4096)[m'] = 0.5 - 0.5*cos(2*pi*m'/4095) (symmetric); the kernel forms the cosine of
    // m' = 256a + m by angle addition from (cos, sin)(2*pi*m/4095) here and the per-a constants below
    win[m].x = (T)cosl(2 * PI * m / 4095.0L);
    win[m].y = (T)sinl(2 * PI * m / 4095.0L);
  }
  V2 wa[16], w32c[8];
  for (int a = 0; a < 16; ++a) {
    wa[a].x = (T)cosl(2 * PI * 256.0L * a / 4095.0L);
    wa[a].y = (T)sinl(2 * PI * 256.0L * a / 4095.0L);
  }
  for (int k = 0; k < 8; ++k) {
    w32c[k].x = (T)cosl(-2 * PI * k / 32.0L);
    w32c[k].y = (T)sinl(-2 * PI * k / 32.0L);
  }
  V2 spc[9];
  for (int i = 0; i < 9; ++i) {
    const int k = i < 5 ? 256 * i : 128 + 256 * (i - 5);
    spc[i].x = (T)cosl(-2 * PI * k / 4096.0L);
    spc[i].y = (T)sinl(-2 * PI * k / 4096.0L);
  }
  if (sizeof(T) == 8) {
    SIA_CUDA(cudaMemcpyToSymbol(c_spc_d, spc, sizeof spc));
    SIA_CUDA(cudaMemcpyToSymbol(c_winA_d, wa, sizeof wa));
    SIA_CUDA(cudaMemcpyToSymbol(c_w32_d, w32c, sizeof w32c));
  } else {
    SIA_CUDA(cudaMemcpyToSymbol(c_spc_f, spc, sizeof spc));
    SIA_CUDA(cudaMemcpyToSymbol(c_winA_f, wa, sizeof wa));
    SIA_CUDA(cudaMemcpyToSymbol(c_w32_f, w32c, sizeof w32c));
  }
  for (int ka = 0; ka < 16; ++ka)
    for (int t = 0; t < 128; ++t) {
      long double ang = -2 * PI * (long double)(t * ka) / 2048.0L;
      twA[ka * 128 + t].x = (T)cosl(ang); twA[ka * 128 + t].y = (T)sinl(ang);
    }
  for (int kb = 0; kb < 16; ++kb)
    for (int c = 0; c < 8; ++c) {
      long double ang = -2 * PI * (long double)(c * kb) / 128.0L;
      twB[kb * 8 + c].x = (T)cosl(ang); twB[kb * 8 + c].y = (T)sinl(ang);
    }
  for (int k = 0; k <= 1024; ++k) {
    long double ang = -2 * PI * (long double)k / 4096.0L;
    twP[k].x = (T)cosl(ang); twP[k].y = (T)sinl(ang);
  }
  const size_t total = (win.size() + twA.size() + twB.size() + twP.size()) * sizeof(V2);
  char *d = nullptr;
  SIA_CUDA(cudaMalloc(&d, total));
  tb.base = d;
  size_t o = 0;
  auto put = [&](const std::vector<V2> &v, const void **dst) -> cudaError_t {
    *dst = d + o;
    cudaError_t e = cudaMemcpy(d + o, v.data(), v.size() * sizeof(V2), cudaMemcpyHostToDevice);
    o += v.size() * sizeof(V2);
    return e;
  };
  SIA_CUDA(put(win, &tb.win2));
  SIA_CUDA(put(twA, &tb.twA));
  SIA_CUDA(put(twB, &tb.twB));
  SIA_CUDA(put(twP, &tb.twP));
  return SIA_OK;
}

int stft_tables_create(StftTables<float> &f, StftTables<double> &d) {
  int rc = upload_tables<float>(f);
  if (rc) return rc;
  return upload_tables<double>(d);
}

void stft_tables_destroy(StftTables<float> &f, StftTables<double> &d) {
  if (f.base) cudaFree(f.base);
  if (d.base) cudaFree(d.base);
  f.base = d.base = nullptr;
}

double hann_power_sum() {
  // sum(np.hanning(4096)**2) accumulated like numpy would to double precision
  const long double PI = 3.141592653589793238462643383279502884L;
  long double s = 0;
  for (int n = 0; n < 4096; ++n) {
    double w = (double)(0.5L - 0.5L * cosl(2 * PI * n / 4095.0L));
    s += (long double)w * w;
  }
  return (double)s;
}

template <typename T, typename OutT>
static int launch(const StftLaunch &a, const StftTables<T> &tb, cudaStream_t s) {
  using V2 = typename Vec2<T>::type;
  // 1/16: the post-pass keeps 2E, 2O (x4 in power) and the window is applied as 2w (x4 in power)
  const double scale = 1.0 / (16.0 * a.Fs * hann_power_sum());
  auto mk = [](double sc) {
    DbScale d;
    const double K = log2(sc);
    d.ke = (int)floor(K) - 1023;
    d.kf = (float)(K - floor(K));
    d.kif = (float)floor(K);
    d.c = 10.0 * log10(sc);
    return d;
  };
  const DbScale sc_edge = mk(scale), sc_mid = mk(2.0 * scale);   // bins 0 and 2048 are not doubled
  const int G = a.frames_per_cta;
  const int64_t blocks = ceil_div(a.total_frames, G);
  if (blocks == 0) return SIA_OK;
  // 80 % of the SM's 228 KB L1/shared storage as shared memory = 182 KB: room for the 4 resident CTAs (4 x 44.5 KB) and
  // ~70 KB of L1 for the twiddle / window tables, which the maximum carveout squeezes out (measured 38.3 ms at 100 %,
  // 36.5 ms at 80 %)
  auto kernel = a.hop == SIA_HOP ? stft_db_kernel<T, OutT, false> : stft_db_kernel<T, OutT, true>;
  SIA_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, 80));
  kernel<<<(unsigned)blocks, 128, 0, s>>>(
      a.d_pcm, a.d_track_starts, a.d_track_len, a.d_frame_starts, a.n_tracks, a.total_frames, G, (OutT *)a.d_spec,
      sc_mid, sc_edge, (const V2 *)tb.win2, (const V2 *)tb.twA, (const V2 *)tb.twB, (const V2 *)tb.twP, a.hop);
  SIA_CHECK_LAUNCH();
  return SIA_OK;
}

int stft_db_launch(const StftLaunch &a, const StftTables<float> &tf, const StftTables<double> &td,
                   cudaStream_t s) {
  if (a.compute == SIA_F64) {
    return a.out_type == SIA_F64 ? launch<double, double>(a, td, s) : launch<double, float>(a, td, s);
  }
  return a.out_type == SIA_F64 ? launch<float, double>(a, tf, s) : launch<float, float>(a, tf, s);
}

}  // namespace sia
