// STFT front end and inverse-STFT overlap-add back end (HBM-bound CUDA-core kernels).
//
// Forward (N_HANS___Selective_Noise/apply.py:142-163, 368-375; reader.py:334-350):
//   peak normalise in float64 -> float32, frames x[160 t : 160 t + 400] * periodic Hann, rfft-400,
//   log(|X| + 1e-5) and angle(X), fused in one kernel (stft_kernel).
// Inverse (SN/apply.py:189-204 = tf.signal.inverse_stft with inverse_stft_window_fn(160, hann)):
//   exp(logmag) e^{j phase} -> irfft-400 -> synthesis window -> 3-frame gather overlap-add ->
//   float32 and/or int16 PCM, fused in one kernel (istft_kernel), no atomics.
//
// FFT-400 is not a power of two (SURVEY.md F3): the real transform is one complex FFT-200 on packed even/odd
// samples, 200 = 8 x 25.  Round 2 layout (round 1 ran three block-wide passes with a __syncthreads after each and was
// issue / latency bound at 0.2 of the HBM roofline): a WARP owns four frames from the samples to the spectrum and
// synchronises with __syncwarp only -
//   pass A   25 radix-8 butterflies per frame (window / pre-twiddle fused), 100 tasks over 32 lanes
//   pass B   8 DFT-25 per frame, each entirely in the registers of one lane (two radix-5 stages, compile-time
//            twiddles): 4 frames x 8 = exactly one task per lane, in place
//   post     bins k and 200 - k of the real transform come from the same two DFT values: 101 pair tasks per frame,
//            lanes walk consecutive bins so that the global stores are coalesced
// One 1.6 KB buffer per frame is the whole working set (pass A and B run in place).  The forward kernel stages the
// int16 span of its 16 frames with one 1-D bulk TMA copy (cp.async.bulk, mbarrier completion) and converts each
// sample once; the inverse kernel gathers 26 output hops from 28 frames and writes 128-bit / 64-bit vectors.
#include "kernels.h"
#include "fft400.cuh"
#include "ptx.cuh"

#include <math.h>
#include <vector>

namespace nhans {

namespace {

constexpr int kWin = 400;
constexpr int kHop = 160;
constexpr int kBinsD = 201;
constexpr int kFW = 4;                  // frames per warp
constexpr int kSW = 4;                  // warps per CTA (forward)
constexpr int kFB = kFW * kSW;          // frames per CTA (forward)
constexpr int kSpanF = (kFB - 1) * kHop + kWin;
constexpr int kIW = 7;                  // warps per CTA (inverse): 28 frames x 1.6 KB stay under the 48 KB static limit
constexpr int kNFI = kFW * kIW;         // frames per CTA (inverse)
constexpr int kOH = kNFI - 2;           // output hops per CTA (2 of 28 frames are recomputed by the neighbour)
constexpr int kThreads = kIW * 32;      // inverse kernels

__device__ float2 g_tw200[200];         // e^{-2 pi i t / 200}
__device__ float2 g_tw400[201];         // e^{-2 pi i k / 400}
__device__ __align__(16) float g_hann[400];           // 0.5 - 0.5 cos(2 pi n / 400)
__device__ __align__(16) float g_winv[400];           // hann[n] / sum_j hann^2[n mod 160 + 160 j] / 400

using namespace fft;

// numpy: abs(int16(-32768)) == -32768, so that sample never wins the max (SN/apply.py:150)
__device__ __forceinline__ int abs16(int v) { return v == -32768 ? -32768 : (v < 0 ? -v : v); }

__global__ void peak_kernel(const int16_t* __restrict__ pcm, const long long* __restrict__ offs, int* __restrict__ peak) {
  const int u = blockIdx.x;
  const long long b = offs[u], e = offs[u + 1];
  int m = -32768;
  for (long long i = b + threadIdx.x; i < e; i += blockDim.x) m = max(m, abs16((int)pcm[i]));
  __shared__ int red[32];
  for (int o = 16; o; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x < 32) {
    m = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : -32768;
    for (int o = 16; o; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (threadIdx.x == 0) peak[u] = (e > b) ? m : 0;
  }
}

// One spectrum value -> log-magnitude and phase (or unit phasor) of bin `o`.
template <bool PHASOR>
__device__ __forceinline__ void emit_bin(float re, float im, int o, float* __restrict__ logmag, float* __restrict__ phase) {
  const float r2 = re * re + im * im;
  if (PHASOR) {
    float inv;
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(inv) : "f"(r2));      // 1 MUFU; r2 = 0 (or denormal) -> inf, replaced below
    inv = r2 > 1e-30f ? inv : 0.f;
    logmag[o] = __logf(r2 * inv + 1e-5f);
    reinterpret_cast<float2*>(phase)[o] = r2 > 1e-30f ? make_float2(re * inv, im * inv) : make_float2(1.f, 0.f);
  } else {
    logmag[o] = __logf(sqrtf(r2) + 1e-5f);
    if (phase) phase[o] = atan2f(im, re);
  }
}

// Pass B of the DFT-200 for the (up to) four frames of a warp, in place: lane = (frame, k1) owns one DFT-25.
template <bool INV>
__device__ __forceinline__ void warp_pass_b(float2* __restrict__ z, int nfw, int lane) {
  const int f = lane >> 3, k1 = lane & 7;
  float2 y[25];
  if (f < nfw) {
    const float2* src = z + f * 200 + k1 * 25;
#pragma unroll
    for (int i = 0; i < 25; ++i) y[i] = src[i];
    dft25<INV>(y);
  }
  __syncwarp();                         // every lane has read its inputs before anyone overwrites them
  if (f < nfw) {
    float2* dst = z + f * 200 + k1;
#pragma unroll
    for (int c = 0; c < 5; ++c)
#pragma unroll
      for (int d = 0; d < 5; ++d) dst[8 * (c + 5 * d)] = y[5 * c + d];
  }
  __syncwarp();
}

// grid: (ceil(max_frames / kFB), U), 128 threads.  PHASOR: the second output is the unit phasor X / |X| as float2
// ((1, 0) where X = 0) instead of the angle - what the fused path keeps between the two transforms (SURVEY.md A.3:
// no atan2 here, no sincos in the inverse).
template <bool PHASOR>
__global__ void __launch_bounds__(kSW * 32, 6)
stft_kernel(const int16_t* __restrict__ pcm, const float* __restrict__ xf, const long long* __restrict__ offs,
            const long long* __restrict__ frame_offs, const int* __restrict__ peak, float* __restrict__ logmag,
            float* __restrict__ phase) {
  __shared__ __align__(16) float s_x[kSpanF];
  __shared__ __align__(16) float2 s_z[kSW][kFW * 200];
  // TMA landing zone of the int16 span (16-byte aligned start and size): the FFT buffers, which nobody touches
  // before the samples are converted
  int16_t* s_raw = reinterpret_cast<int16_t*>(&s_z[0][0]);
  static_assert(sizeof(float2) * kSW * kFW * 200 >= (kSpanF + 16) * sizeof(int16_t), "raw span must fit the FFT buffers");
  __shared__ __align__(8) uint64_t s_bar;
  const int u = blockIdx.y;
  const int T = (int)(frame_offs[u + 1] - frame_offs[u]);
  const int t0 = blockIdx.x * kFB;
  if (t0 >= T) return;
  const int nf = min(kFB, T - t0);
  const long long base = offs[u] + (long long)t0 * kHop;
  const int span = (nf - 1) * kHop + kWin;
  if (xf) {                              // already-normalised float samples (apply_demo, SN/apply.py:241-247)
    for (int i = threadIdx.x; i < span; i += blockDim.x) s_x[i] = xf[base + i];
  } else {
    // one bulk copy of the int16 span, from the 16-byte boundary below its first sample
    const long long abase = base & ~7LL;
    const int shift = (int)(base - abase);
    const uint32_t bytes = (uint32_t)(((shift + span) * 2 + 15) & ~15);
    if (threadIdx.x == 0) {
      ptx::mbar_init(&s_bar, 1);
      ptx::fence_barrier_init();
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      ptx::mbar_expect_tx(&s_bar, bytes);
      ptx::bulk_load_1d(s_raw, pcm + abase, bytes, &s_bar);
    }
    ptx::mbar_wait(&s_bar, 0, nullptr, 7);          // bounded: traps instead of hanging if the copy never lands
    // x / (peak + 1e-6) in float64 like the reference, as a multiplication by the float64 reciprocal (differs from
    // the true quotient by < 1 float64 ulp before the rounding to float32; nhans_normalise keeps the exact division)
    const double inv = 1.0 / ((double)peak[u] + 0.000001);
    for (int i = threadIdx.x; i < span; i += blockDim.x) s_x[i] = (float)((double)s_raw[shift + i] * inv);
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nfw = min(kFW, nf - warp * kFW);          // frames of this warp
  if (nfw <= 0) return;
  float2* z = s_z[warp];
  const float* x0 = s_x + warp * kFW * kHop;
  // pass A on the windowed, even/odd-packed samples z[m] = (x[2m] w[2m], x[2m+1] w[2m+1]), m = 25 m1 + m2
  for (int t = lane, f = lane >= 25, m2 = lane - 25 * f; t < nfw * 25; t += 32) {
    float2 v[8];
#pragma unroll
    for (int m1 = 0; m1 < 8; ++m1) {
      const int m = 25 * m1 + m2;
      const float2 xx = *reinterpret_cast<const float2*>(&x0[f * kHop + 2 * m]);
      const float2 h = __ldg(reinterpret_cast<const float2*>(g_hann) + m);
      v[m1] = cmul2(xx, h);
    }
    dft8<false>(v);
    z[f * 200 + m2] = v[0];
    // W200^{m2 k1}, k1 = 1..7, as powers of one table value (7 scattered table reads per task kept the L1 data pipe
    // at 68 % in round 2's first version; 6 complex multiplies are cheaper)
    const float2 w1 = __ldg(&g_tw200[m2]);
    float2 w = w1;
#pragma unroll
    for (int k1 = 1; k1 < 8; ++k1) {
      z[f * 200 + k1 * 25 + m2] = cmul(v[k1], w);
      if (k1 < 7) w = cmul(w, w1);
    }
    m2 += 7; f += 1;                     // t + 32 = 25 (f + 1) + (m2 + 7)
    if (m2 >= 25) { m2 -= 25; f += 1; }
  }
  __syncwarp();
  warp_pass_b<false>(z, nfw, lane);
  // bins k and 200 - k from Z[k], Z[200 - k]:  with E = (Z[k] + conj Z[200-k]) / 2, P = e^{-2 pi i k / 400} (Z[k] - conj Z[200-k]) / 2:
  //   X[k] = E - i P,   X[200 - k] = conj(E) - i conj(P)
  const long long row0 = frame_offs[u] + t0 + warp * kFW;
  float* lm_w = logmag + (size_t)row0 * kBinsD;                       // 32-bit offsets from the warp's first row
  float* ph_w = phase ? phase + (size_t)row0 * kBinsD * (PHASOR ? 2 : 1) : nullptr;
  float2 w_next = __ldg(&g_tw400[lane]);                              // table value of the next iteration: off the critical path
  for (int i = lane, f = 0, k = lane; i < nfw * 101; i += 32) {
    const float2 a = z[f * 200 + k];
    const float2 b = z[f * 200 + (k ? 200 - k : 0)];
    const float2 w = w_next;
    w_next = __ldg(&g_tw400[k + 32 >= 101 ? k + 32 - 101 : k + 32]);
    const float2 cb = cconj(b);
    const float2 E = cscale(cadd(a, cb), 0.5f), O = cscale(csub(a, cb), 0.5f);
    const float2 P = cmul(w, O);
    const float2 Xk = cadd(E, rot<false>(P));                        // E - i P
    const float2 Xm = csub(cconj(E), make_float2(P.y, P.x));         // conj(E) - i conj(P)
    const int o = f * kBinsD;
    emit_bin<PHASOR>(Xk.x, Xk.y, o + k, lm_w, ph_w);
    if (k != 100) emit_bin<PHASOR>(Xm.x, Xm.y, o + 200 - k, lm_w, ph_w);
    k += 32;
    if (k >= 101) { k -= 101; f += 1; }
  }
}

// Normalised (and, for the mixture, trimmed) float32 samples: stage a2 on its own, for the bit-exact test.
__global__ void normalise_kernel(const int16_t* __restrict__ pcm, const long long* __restrict__ offs,
                                 const long long* __restrict__ out_offs, const int* __restrict__ peak, float* __restrict__ out) {
  const int u = blockIdx.y;
  const long long n = out_offs[u + 1] - out_offs[u];
  const double denom = (double)peak[u] + 0.000001;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    out[out_offs[u] + i] = (float)((double)pcm[offs[u] + i] / denom);
}

// exp(logmag) e^{j phase} -> irfft-400 -> synthesis window for frames fa .. fa + kNFI - 1 of clip rows
// [row0, row0 + T); leaves the windowed frames in s_y[kNFI][400] (frames outside the clip are zero).
// PHASOR: `phase` holds unit phasors (float2) instead of angles.  Every warp transforms its own four frames;
// the block synchronises once at the end (and once at the start: the buffer may still be read by the caller).
template <bool PHASOR>
__device__ __forceinline__ void istft_frames(float* __restrict__ s_y, const float* __restrict__ logmag,
                                             const float* __restrict__ phase, long long row0, int T, int fa) {
  __syncthreads();                         // previous use of the buffer is over
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float2* z = reinterpret_cast<float2*>(s_y) + warp * kFW * 200;
  const int t_first = fa + warp * kFW;
  // The warp's four spectrum rows are contiguous in HBM (4 x 804 B of log-magnitudes, 4 x 1608 B of phasors): ask L2 for
  // all of their lines first (no registers held), then read them in batches of kLB iterations with every load of a
  // batch issued before the first use.  One element per iteration with the use right behind the load left the warp on
  // a long-scoreboard stall for 44 % of its samples (ncu source page, round 2).
  {
    const int ta = max(t_first, 0), tb = min(t_first + kFW, T);
    if (tb > ta) {
      const char* l0 = reinterpret_cast<const char*>(logmag + (size_t)(row0 + ta) * kBinsD);
      const char* p0 = reinterpret_cast<const char*>(phase + (size_t)(row0 + ta) * kBinsD * (PHASOR ? 2 : 1));
      const int lbytes = (tb - ta) * kBinsD * 4, pbytes = lbytes * (PHASOR ? 2 : 1);
      for (int o = lane * 128; o < lbytes; o += 32 * 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(l0 + o));
      for (int o = lane * 128; o < pbytes; o += 32 * 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(p0 + o));
    }
  }
  // S[k] = exp(logmag) * phasor; Z[k] = (S[k] + conj S[200-k]) + i e^{+2 pi i k / 400} (S[k] - conj S[200-k]) and
  // Z[200 - k] from the same pair
  constexpr int kLoadIts = (kFW * 101 + 31) / 32, kLB = 4;
#pragma unroll
  for (int j0 = 0; j0 < kLoadIts; j0 += kLB) {
    float lk[kLB], lm[kLB];
    float2 pk[kLB], pm[kLB], w[kLB];
    bool ok[kLB];
#pragma unroll
    for (int j = 0; j < kLB; ++j) {
      const int i = lane + 32 * (j0 + j);
      const int f = i / 101, k = i - 101 * f;
      const int t = t_first + f;
      ok[j] = j0 + j < kLoadIts && i < kFW * 101 && t >= 0 && t < T;
      lk[j] = lm[j] = 0.f;
      pk[j] = pm[j] = make_float2(0.f, 0.f);
      if (ok[j]) {
        const size_t o = (size_t)(row0 + t) * kBinsD;
        lk[j] = logmag[o + k];
        lm[j] = logmag[o + 200 - k];
        if (PHASOR) {
          pk[j] = reinterpret_cast<const float2*>(phase)[o + k];
          pm[j] = reinterpret_cast<const float2*>(phase)[o + 200 - k];
        } else {
          pk[j].x = phase[o + k];
          pm[j].x = phase[o + 200 - k];
        }
      }
      w[j] = __ldg(&g_tw400[i < kFW * 101 ? k : 0]);     // conj(w) = e^{+2 pi i k / 400}
    }
#pragma unroll
    for (int j = 0; j < kLB; ++j) {
      const int i = lane + 32 * (j0 + j);
      if (j0 + j >= kLoadIts || i >= kFW * 101) continue;
      const int f = i / 101, k = i - 101 * f;
      float2 sk = make_float2(0.f, 0.f), sm = sk;
      if (ok[j]) {
        // __expf: 2 ulp, i.e. ~1e-6 relative on |S| - far inside the 1e-5 absolute bound of the waveform tests
        const float ak = __expf(lk[j]), am = __expf(lm[j]);
        if (PHASOR) {
          sk = cscale(pk[j], ak);
          sm = cscale(pm[j], am);
        } else {
          float sn, cs;
          sincosf(pk[j].x, &sn, &cs);
          sk = make_float2(ak * cs, ak * sn);
          sincosf(pm[j].x, &sn, &cs);
          sm = make_float2(am * cs, am * sn);
        }
        if (k == 0) { sk.y = 0.f; sm.y = 0.f; }           // irfft ignores the imaginary part of DC / Nyquist
      }
      const float2 cm = cconj(sm);
      const float2 e = cadd(sk, cm), d = csub(sk, cm);
      const float2 wd = cmul(cconj(w[j]), d);
      z[f * 200 + k] = cadd(e, rot<true>(wd));                                  // e + i wd
      if (k > 0 && k < 100) z[f * 200 + 200 - k] = cadd(cconj(e), make_float2(wd.y, wd.x));
    }
  }
  __syncwarp();
  // pass A in place: task (f, m2) reads and writes the slots 25 j + m2
  for (int t = lane, f = lane >= 25, m2 = lane - 25 * f; t < kFW * 25; t += 32) {
    float2 v[8];
#pragma unroll
    for (int m1 = 0; m1 < 8; ++m1) v[m1] = z[f * 200 + 25 * m1 + m2];
    dft8<true>(v);
    z[f * 200 + m2] = v[0];
    const float2 w1 = cconj(__ldg(&g_tw200[m2]));
    float2 w = w1;
#pragma unroll
    for (int k1 = 1; k1 < 8; ++k1) {
      z[f * 200 + k1 * 25 + m2] = cmul(v[k1], w);
      if (k1 < 7) w = cmul(w, w1);
    }
    m2 += 7; f += 1;                     // t + 32 = 25 (f + 1) + (m2 + 7)
    if (m2 >= 25) { m2 -= 25; f += 1; }
  }
  __syncwarp();
  warp_pass_b<true>(z, kFW, lane);
  // frames: y_f[2m] = Re z[m] / 400, y_f[2m+1] = Im z[m] / 400, times the synthesis window
  for (int i = lane, m = lane; i < kFW * 200; i += 32) {
    const float2 v = z[i];
    const float2 w = __ldg(reinterpret_cast<const float2*>(g_winv) + m);
    z[i] = cmul2(v, w);                                  // g_winv carries the 1 / 400 of the inverse transform
    m += 32;
    if (m >= 200) m -= 200;
  }
  __syncthreads();
}

// 3-frame gather overlap-add of samples i .. i + 3 of the block (i % 4 == 0, so all four lie in hop hl = i / 160)
__device__ __forceinline__ float4 ola_sample4(const float* s_y, int i) {
  const int hl = i / kHop, r = i - hl * kHop;
  // frame local index f = hl + 2 - j covers sample offset r + 160 j, j = 0..2 (zero frames outside [0, T))
  const float4 a = *reinterpret_cast<const float4*>(&s_y[(hl + 2) * kWin + r]);
  const float4 b = *reinterpret_cast<const float4*>(&s_y[(hl + 1) * kWin + r + kHop]);
  float4 acc = make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
  if (r + 2 * kHop < kWin) {
    const float4 c = *reinterpret_cast<const float4*>(&s_y[hl * kWin + r + 2 * kHop]);
    acc.x += c.x; acc.y += c.y; acc.z += c.z; acc.w += c.w;
  }
  return acc;
}

__device__ __forceinline__ int16_t to_i16(float v) { return (int16_t)__float2int_rn(fminf(fmaxf(v, -32768.f), 32767.f)); }

// Samples o .. o + 3 as float32 and / or int16 PCM (v * scale, peak de-normalised); either output may be null
__device__ __forceinline__ void store4(float* out_f32, int16_t* out_i16, long long o, float4 v, float scale) {
  if (out_f32) *reinterpret_cast<float4*>(out_f32 + o) = v;
  if (out_i16) {
    short4 q;
    q.x = to_i16(v.x * scale); q.y = to_i16(v.y * scale); q.z = to_i16(v.z * scale); q.w = to_i16(v.w * scale);
    *reinterpret_cast<short4*>(out_i16 + o) = q;
  }
}

// grid: (ceil((max_frames + 2) / kOH), U).  Output hop h (160 samples) sums frames h-2, h-1, h.  Clip lengths and
// hop starts are multiples of 80 samples, so groups of four samples are aligned for 128-bit (f32) / 64-bit (int16) stores.
template <bool PHASOR>
__global__ void __launch_bounds__(kThreads, 4)
istft_kernel(const float* __restrict__ logmag, const float* __restrict__ phase, const long long* __restrict__ frame_offs,
             const long long* __restrict__ out_offs, const int* __restrict__ peak, float* __restrict__ out_f32,
             int16_t* __restrict__ out_i16) {
  __shared__ __align__(16) float s_y[kNFI * kWin];
  const int u = blockIdx.y;
  const int T = (int)(frame_offs[u + 1] - frame_offs[u]);
  if (T <= 0) return;
  const int h0 = blockIdx.x * kOH;        // first output hop
  if (h0 >= T + 2) return;
  istft_frames<PHASOR>(s_y, logmag, phase, frame_offs[u], T, h0 - 2);
  const long long n_out = out_offs[u + 1] - out_offs[u];   // (T - 1) * 160 + 400
  const float scale = (float)((double)peak[u] + 0.000001);
  for (int i = threadIdx.x * 4; i < kOH * kHop; i += blockDim.x * 4) {
    const long long n = (long long)h0 * kHop + i;
    if (n >= n_out) break;
    store4(out_f32, out_i16, out_offs[u] + n, ola_sample4(s_y, i), scale);
  }
}

// The same inverse STFT over the segments of a stream step (kernels.h StreamStepDev): local frame 0 of stream s is
// the first carried denoised frame (den_carry of them precede its windows), frames outside [0, T) are zero as at an
// utterance edge, and local samples [lo, lo + len) with lo = 160 den_carry go to out_offs[s].  Every sample is the same
// gather and sum as in istft_kernel, so a stream's samples are bit-identical to the whole clip's.
// POST adds the post-mix outputs of istft_post_kernel / compensate_kernel: the same rows of seg_lm (the input spectrum,
// with the same phasors) give mixed_processed, then removed = mixed - den, compensated = den + removed * factor[s], and
// the energy sums of den and removed go to sums[s][0..1] (zeroed by the launcher).  Any output may be null.
// grid: (ceil((max len + 159) / 160 / kOH), n).
template <bool POST>
__global__ void __launch_bounds__(kThreads, POST ? 1 : 4)
istft_stream_kernel(const StreamStepDev p, float* __restrict__ out_f32, int16_t* __restrict__ out_i16, float* __restrict__ mixed_f32,
                    float* __restrict__ removed_f32, float* __restrict__ comp_f32, const float* __restrict__ factor,
                    double* __restrict__ sums /* [n][2] */) {
  __shared__ __align__(16) float s_y[kNFI * kWin];
  const int u = blockIdx.y;
  const int dc = p.den_carry[u];
  const int T = dc + (int)(p.win_offs[u + 1] - p.win_offs[u]);
  const long long len = p.out_offs[u + 1] - p.out_offs[u];
  const int h0 = dc + blockIdx.x * kOH;   // first output hop (local)
  if (T <= 0 || (long long)blockIdx.x * kOH * kHop >= len) return;
  const long long row0 = p.seg_offs[u] + p.left[u] - dc;
  istft_frames<true>(s_y, p.den_seg, p.seg_ph, row0, T, h0 - 2);
  const long long lo = (long long)dc * kHop;
  const float scale = (float)((double)p.peak[u] + 0.000001);
  if constexpr (!POST) {
    for (int i = threadIdx.x * 4; i < kOH * kHop; i += blockDim.x * 4) {
      const long long n = (long long)h0 * kHop + i - lo;
      if (n >= len) break;
      const float4 acc = ola_sample4(s_y, i);
      store4(out_f32, out_i16, p.out_offs[u] + n, acc, scale);
    }
  } else {
    __shared__ float s_red[2][kThreads / 32];
    constexpr int PER = (kOH * kHop / 4 + kThreads - 1) / kThreads;
    float4 den[PER];
#pragma unroll
    for (int k = 0; k < PER; ++k) {
      const int i = (threadIdx.x + k * kThreads) * 4;
      den[k] = i < kOH * kHop ? ola_sample4(s_y, i) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    istft_frames<true>(s_y, p.seg_lm, p.seg_ph, row0, T, h0 - 2);
    const float f = factor[u];
    float e_den = 0.f, e_rem = 0.f;
#pragma unroll
    for (int k = 0; k < PER; ++k) {
      const int i = (threadIdx.x + k * kThreads) * 4;
      const long long n = (long long)h0 * kHop + i - lo;
      if (i >= kOH * kHop || n >= len) continue;
      const float4 mixed = ola_sample4(s_y, i);
      const float4 d = den[k];
      const float4 rem = make_float4(mixed.x - d.x, mixed.y - d.y, mixed.z - d.z, mixed.w - d.w);
      const long long o = p.out_offs[u] + n;
      store4(out_f32, out_i16, o, d, scale);
      if (mixed_f32) *reinterpret_cast<float4*>(mixed_f32 + o) = mixed;
      if (removed_f32) *reinterpret_cast<float4*>(removed_f32 + o) = rem;
      // one FFMA per sample, as compensate_kernel's den + removed * factor
      if (comp_f32)
        *reinterpret_cast<float4*>(comp_f32 + o) = make_float4(__fmaf_rn(rem.x, f, d.x), __fmaf_rn(rem.y, f, d.y),
                                                               __fmaf_rn(rem.z, f, d.z), __fmaf_rn(rem.w, f, d.w));
      e_den += d.x * d.x + d.y * d.y + d.z * d.z + d.w * d.w;
      e_rem += rem.x * rem.x + rem.y * rem.y + rem.z * rem.z + rem.w * rem.w;
    }
    for (int o = 16; o; o >>= 1) {
      e_den += __shfl_xor_sync(0xffffffffu, e_den, o);
      e_rem += __shfl_xor_sync(0xffffffffu, e_rem, o);
    }
    if ((threadIdx.x & 31) == 0) { s_red[0][threadIdx.x >> 5] = e_den; s_red[1][threadIdx.x >> 5] = e_rem; }
    __syncthreads();
    if (threadIdx.x == 0) {
      double a = 0, b = 0;
      for (int w = 0; w < kThreads / 32; ++w) { a += s_red[0][w]; b += s_red[1][w]; }
      atomicAdd(&sums[2 * u], a);
      atomicAdd(&sums[2 * u + 1], b);
    }
  }
}

// Post-mix outputs of apply_snc (SN/apply.py:456-464) fused into one pass: both inverse STFTs (denoised
// spectrum and the input spectrum = 'mixed_processed'), removed = mixed_processed - denoised, and the two
// per-clip energy sums of snr_est = mean(denoised^2) / mean(removed^2).
__global__ void __launch_bounds__(kThreads)
istft_post_kernel(const float* __restrict__ den_logmag, const float* __restrict__ mix_logmag, const float* __restrict__ phase,
                  const long long* __restrict__ frame_offs, const long long* __restrict__ out_offs,
                  float* __restrict__ den_f32, float* __restrict__ mixed_f32, float* __restrict__ removed_f32,
                  double* __restrict__ sums /* [U][2] */) {
  __shared__ __align__(16) float s_y[kNFI * kWin];
  __shared__ float s_red[2][kThreads / 32];
  const int u = blockIdx.y;
  const int T = (int)(frame_offs[u + 1] - frame_offs[u]);
  if (T <= 0) return;
  const int h0 = blockIdx.x * kOH;
  if (h0 >= T + 2) return;
  constexpr int PER = (kOH * kHop / 4 + kThreads - 1) / kThreads;
  float4 den[PER];
  istft_frames<true>(s_y, den_logmag, phase, frame_offs[u], T, h0 - 2);
#pragma unroll
  for (int k = 0; k < PER; ++k) {
    const int i = (threadIdx.x + k * kThreads) * 4;
    den[k] = i < kOH * kHop ? ola_sample4(s_y, i) : make_float4(0.f, 0.f, 0.f, 0.f);
  }
  istft_frames<true>(s_y, mix_logmag, phase, frame_offs[u], T, h0 - 2);
  const long long n_out = out_offs[u + 1] - out_offs[u];
  float e_den = 0.f, e_rem = 0.f;
#pragma unroll
  for (int k = 0; k < PER; ++k) {
    const int i = (threadIdx.x + k * kThreads) * 4;
    const long long n = (long long)h0 * kHop + i;
    if (i >= kOH * kHop || n >= n_out) continue;
    const float4 mixed = ola_sample4(s_y, i);
    const float4 d = den[k];
    const float4 rem = make_float4(mixed.x - d.x, mixed.y - d.y, mixed.z - d.z, mixed.w - d.w);     // SN/apply.py:460
    const long long o = out_offs[u] + n;
    if (den_f32) *reinterpret_cast<float4*>(den_f32 + o) = d;
    if (mixed_f32) *reinterpret_cast<float4*>(mixed_f32 + o) = mixed;
    if (removed_f32) *reinterpret_cast<float4*>(removed_f32 + o) = rem;
    e_den += d.x * d.x + d.y * d.y + d.z * d.z + d.w * d.w;
    e_rem += rem.x * rem.x + rem.y * rem.y + rem.z * rem.z + rem.w * rem.w;
  }
  for (int o = 16; o; o >>= 1) {
    e_den += __shfl_xor_sync(0xffffffffu, e_den, o);
    e_rem += __shfl_xor_sync(0xffffffffu, e_rem, o);
  }
  if ((threadIdx.x & 31) == 0) { s_red[0][threadIdx.x >> 5] = e_den; s_red[1][threadIdx.x >> 5] = e_rem; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double a = 0, b = 0;
    for (int w = 0; w < kThreads / 32; ++w) { a += s_red[0][w]; b += s_red[1][w]; }
    atomicAdd(&sums[2 * u], a);
    atomicAdd(&sums[2 * u + 1], b);
  }
}

// compensated = denoised + removed * factor, factor = snr_est / 20 (--ac) or the --compensate constant
// (SN/apply.py:466-470); also writes snr_est[u].
__global__ void compensate_kernel(const float* __restrict__ den, const float* __restrict__ removed,
                                  const long long* __restrict__ out_offs, const double* __restrict__ sums, float compensate, int ac,
                                  float* __restrict__ out, float* __restrict__ snr_est) {
  const int u = blockIdx.y;
  const long long b = out_offs[u], n = out_offs[u + 1] - b;
  // both means share the sample count, so snr_est is the ratio of the sums
  const double snr = sums[2 * u + 1] > 0 ? sums[2 * u] / sums[2 * u + 1] : INFINITY;
  float factor = ac ? (float)(snr / 20.0) : compensate;
  if (!isfinite(factor)) factor = 0.f;
  if (blockIdx.x == 0 && threadIdx.x == 0 && snr_est) snr_est[u] = (float)snr;
  if (!out) return;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    out[b + i] = den[b + i] + removed[b + i] * factor;
}

// example_loss of the model graph (SN/main.py:243-246): one warp per frame, weights linspace(2, 1, 201)
__global__ void eval_loss_kernel(const float* __restrict__ den, const float* __restrict__ tgt, long long n, float* __restrict__ loss) {
  const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= n) return;
  const int lane = threadIdx.x & 31;
  float acc = 0.f;
  for (int k = lane; k < kBinsD; k += 32) {
    const float d = den[row * kBinsD + k] - tgt[row * kBinsD + k];
    acc += d * d * (2.0f - (float)k * (1.0f / 200.0f));
  }
  for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) loss[row] = acc * (1.0f / 201.0f);
}

}  // namespace

cudaError_t launch_eval_loss(cudaStream_t s, const float* den, const float* tgt, long long n, float* loss) {
  if (n <= 0) return cudaSuccess;
  eval_loss_kernel<<<(unsigned)((n + 7) / 8), 256, 0, s>>>(den, tgt, n, loss);
  return cudaGetLastError();
}

cudaError_t dsp_init_tables() {
  const double kPi = 3.14159265358979323846;
  std::vector<float2> t200(200), t400(201);
  std::vector<float> hann(400), winv(400);
  for (int i = 0; i < 200; ++i) t200[i] = make_float2((float)cos(2 * kPi * i / 200), (float)-sin(2 * kPi * i / 200));
  for (int i = 0; i < 201; ++i) t400[i] = make_float2((float)cos(2 * kPi * i / 400), (float)-sin(2 * kPi * i / 400));
  for (int i = 0; i < 400; ++i) hann[i] = (float)(0.5 - 0.5 * cos(2 * kPi * i / 400));
  for (int i = 0; i < 400; ++i) {
    double d = 0;
    for (int j = 0; j < 3; ++j) {
      int n = (i % 160) + 160 * j;
      if (n < 400) d += (double)hann[n] * (double)hann[n];
    }
    winv[i] = (float)((double)hann[i] / d / 400.0);       // synthesis window x the 1 / N of the unnormalised inverse DFT
  }
  cudaError_t e;
  if ((e = cudaMemcpyToSymbol(g_tw200, t200.data(), sizeof(float2) * 200)) != cudaSuccess) return e;
  if ((e = cudaMemcpyToSymbol(g_tw400, t400.data(), sizeof(float2) * 201)) != cudaSuccess) return e;
  if ((e = cudaMemcpyToSymbol(g_hann, hann.data(), sizeof(float) * 400)) != cudaSuccess) return e;
  if ((e = cudaMemcpyToSymbol(g_winv, winv.data(), sizeof(float) * 400)) != cudaSuccess) return e;
  return cudaSuccess;
}

cudaError_t launch_peaks(cudaStream_t s, const int16_t* pcm, const long long* offs, int U, int* peak) {
  if (U <= 0) return cudaSuccess;
  peak_kernel<<<U, 1024, 0, s>>>(pcm, offs, peak);
  return cudaGetLastError();
}

cudaError_t launch_stft(cudaStream_t s, const int16_t* pcm, const long long* offs, const long long* frame_offs, int U,
                        const int* peak, int max_frames_per_clip, float* logmag, float* phase, bool phasor) {
  if (U <= 0 || max_frames_per_clip <= 0) return cudaSuccess;
  dim3 grid((max_frames_per_clip + kFB - 1) / kFB, U);
  if (phasor) stft_kernel<true><<<grid, kSW * 32, 0, s>>>(pcm, nullptr, offs, frame_offs, peak, logmag, phase);
  else stft_kernel<false><<<grid, kSW * 32, 0, s>>>(pcm, nullptr, offs, frame_offs, peak, logmag, phase);
  return cudaGetLastError();
}

cudaError_t launch_stft_f32(cudaStream_t s, const float* x, const long long* offs, const long long* frame_offs, int U,
                            int max_frames_per_clip, float* logmag, float* phase, bool phasor) {
  if (U <= 0 || max_frames_per_clip <= 0) return cudaSuccess;
  dim3 grid((max_frames_per_clip + kFB - 1) / kFB, U);
  if (phasor) stft_kernel<true><<<grid, kSW * 32, 0, s>>>(nullptr, x, offs, frame_offs, nullptr, logmag, phase);
  else stft_kernel<false><<<grid, kSW * 32, 0, s>>>(nullptr, x, offs, frame_offs, nullptr, logmag, phase);
  return cudaGetLastError();
}

cudaError_t launch_normalise(cudaStream_t s, const int16_t* pcm, const long long* offs, const long long* out_offs, int U,
                             const int* peak, float* out) {
  if (U <= 0) return cudaSuccess;
  dim3 grid(64, U);
  normalise_kernel<<<grid, 256, 0, s>>>(pcm, offs, out_offs, peak, out);
  return cudaGetLastError();
}

cudaError_t launch_istft(cudaStream_t s, const float* logmag, const float* phase, const long long* frame_offs,
                         const long long* out_offs, int U, const int* peak, int max_frames_per_clip, float* out_f32,
                         int16_t* out_i16, bool phasor) {
  if (U <= 0 || max_frames_per_clip <= 0) return cudaSuccess;
  dim3 grid((max_frames_per_clip + 2 + kOH - 1) / kOH, U);
  if (phasor) istft_kernel<true><<<grid, kThreads, 0, s>>>(logmag, phase, frame_offs, out_offs, peak, out_f32, out_i16);
  else istft_kernel<false><<<grid, kThreads, 0, s>>>(logmag, phase, frame_offs, out_offs, peak, out_f32, out_i16);
  return cudaGetLastError();
}

cudaError_t launch_istft_stream(cudaStream_t s, const StreamStepDev& p, int max_samples, float* out_f32, int16_t* out_i16) {
  if (p.n <= 0 || max_samples <= 0) return cudaSuccess;
  dim3 grid((max_samples + kOH * kHop - 1) / (kOH * kHop), p.n);
  istft_stream_kernel<false><<<grid, kThreads, 0, s>>>(p, out_f32, out_i16, nullptr, nullptr, nullptr, nullptr, nullptr);
  return cudaGetLastError();
}

cudaError_t launch_istft_stream_post(cudaStream_t s, const StreamStepDev& p, int max_samples, const float* factor, float* out_f32,
                                     int16_t* out_i16, float* mixed_f32, float* removed_f32, float* comp_f32, double* sums) {
  if (p.n <= 0) return cudaSuccess;
  // zeroed even when the step emits nothing: the caller adds the sums of every stream to its running totals
  cudaError_t e = cudaMemsetAsync(sums, 0, sizeof(double) * 2 * p.n, s);
  if (e != cudaSuccess || max_samples <= 0) return e;
  dim3 grid((max_samples + kOH * kHop - 1) / (kOH * kHop), p.n);
  istft_stream_kernel<true><<<grid, kThreads, 0, s>>>(p, out_f32, out_i16, mixed_f32, removed_f32, comp_f32, factor, sums);
  return cudaGetLastError();
}

cudaError_t launch_istft_post(cudaStream_t s, const float* den_logmag, const float* mix_logmag, const float* phase,
                              const long long* frame_offs, const long long* out_offs, int U, int max_frames_per_clip,
                              float* den_f32, float* mixed_f32, float* removed_f32, double* sums) {
  if (U <= 0) return cudaSuccess;
  // zeroed even when no clip has a frame: compensate_kernel reads the sums of every clip
  cudaError_t e = cudaMemsetAsync(sums, 0, sizeof(double) * 2 * U, s);
  if (e != cudaSuccess || max_frames_per_clip <= 0) return e;
  dim3 grid((max_frames_per_clip + 2 + kOH - 1) / kOH, U);
  istft_post_kernel<<<grid, kThreads, 0, s>>>(den_logmag, mix_logmag, phase, frame_offs, out_offs, den_f32, mixed_f32, removed_f32, sums);
  return cudaGetLastError();
}

cudaError_t launch_compensate(cudaStream_t s, const float* den, const float* removed, const long long* out_offs, int U,
                              const double* sums, float compensate, int ac, float* out, float* snr_est) {
  if (U <= 0) return cudaSuccess;
  dim3 grid(64, U);
  compensate_kernel<<<grid, 256, 0, s>>>(den, removed, out_offs, sums, compensate, ac, out, snr_est);
  return cudaGetLastError();
}

}  // namespace nhans
