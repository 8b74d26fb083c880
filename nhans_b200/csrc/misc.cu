// CUDA-core kernels around the tensor-core GEMMs: the Cin = 1 convolutions (per-frame evaluation + window
// expansion for the mask network, per-unit kernels with the implicit window gather for the towers / fallback), the conditioning-projection table, the tower's global mean pool and the
// per-unit lookup tables.
#include "kernels.h"

namespace nhans {

namespace {

__device__ __forceinline__ uint32_t pack_half2(float a, float b) {
  __half2 h = __floats2half2_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}

// resblock1_1_conv1 (main.py:162, Cin = 1, 4x4) and embedding/noise_resblock1_1_conv1 (main.py:104, 8x4,
// stride 3x2): one thread per output pixel, 64 output channels in registers.  Input row r of unit n is
// frame units.frame[n] + r + raw_oh of the fp32 log-magnitude array; rows outside the clip and outside
// [0, Hin) read 0.0, which is the zero padding of pad_1D_for_windowing (SN/apply.py:170-173) and of the
// 'SAME' convolution at once - the [T, 35, 201] window tensor is never materialised.
constexpr int kDirectPitch = 68;                       // floats per staged pixel row (64 + 4: conflict-free float4 access)
__global__ void __launch_bounds__(128)
direct_conv64_kernel(const DirectDev p) {
  extern __shared__ float s_w[];                       // [kh*kw][64] | 4 x [32][kDirectPitch] staging | metadata
  const int taps = p.kh * p.kw;
  float* s_stage = s_w + taps * 64;
  int* s_meta = reinterpret_cast<int*>(s_stage + 4 * 32 * kDirectPitch);
  for (int i = threadIdx.x; i < taps * 64; i += blockDim.x) s_w[i] = p.w[i];
  __syncthreads();
  const long long total = (long long)p.units * p.Ho * p.Wo;
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const bool valid = idx < total;
  if (!valid) idx = total - 1;                          // tail threads compute a duplicate and store nothing
  const int unit = (int)(idx / (p.Ho * p.Wo));
  const int rem = (int)(idx - (long long)unit * p.Ho * p.Wo);
  const int ho = rem / p.Wo, wo = rem - ho * p.Wo;
  const int frame0 = p.units_tab.frame[unit] + p.raw_oh;
  const int lo = p.units_tab.lo[unit], hi = p.units_tab.hi[unit];
  const EpiDev& e = p.epi;

  float acc[64];
#pragma unroll
  for (int n = 0; n < 64; ++n) acc[n] = 0.f;
  for (int i = 0; i < p.kh; ++i) {
    const int r = ho * p.sh + i - p.pt;
    const int frame = frame0 + r;
    if (r < 0 || r >= p.Hin || frame < lo || frame >= hi) continue;
    const float* row = e.raw + (size_t)frame * 201;
    for (int j = 0; j < p.kw; ++j) {
      const int f = wo * p.sw + j - p.pl;
      if (f < 0 || f >= p.Win) continue;
      const float x = row[f];
      const float4* w4 = reinterpret_cast<const float4*>(s_w + (i * p.kw + j) * 64);
#pragma unroll
      for (int n = 0; n < 16; ++n) {
        const float4 w = w4[n];
        acc[4 * n] = fmaf(x, w.x, acc[4 * n]);
        acc[4 * n + 1] = fmaf(x, w.y, acc[4 * n + 1]);
        acc[4 * n + 2] = fmaf(x, w.z, acc[4 * n + 2]);
        acc[4 * n + 3] = fmaf(x, w.w, acc[4 * n + 3]);
      }
    }
  }
  // Epilogue through a warp-private shared-memory transpose: 8 lanes then cover one pixel's 64 channels, so
  // the table loads and the fp16 stores of a warp touch whole 128-byte lines instead of 32 scattered ones.
  const int utt = p.units_tab.utt ? p.units_tab.utt[unit] : 0;
  const int yy = ho + e.o_oy, xx = wo + e.o_ox;
  const int plane = (yy % e.o_sh) * e.o_sw + (xx % e.o_sw);
  const long long pix = plane * e.o_plane + unit * e.o_ustride + (yy / e.o_sh) * e.o_rstride + (xx / e.o_sw);
  const int lane = threadIdx.x & 31;
  float* st = s_stage + (threadIdx.x >> 5) * (32 * kDirectPitch);
  long long* s_pix = reinterpret_cast<long long*>(s_meta) + (threadIdx.x >> 5) * 32;
  int* s_tf = s_meta + 2 * 4 * 32 + (threadIdx.x >> 5) * 64;
  __syncwarp();
#pragma unroll
  for (int n = 0; n < 16; ++n)
    *reinterpret_cast<float4*>(st + lane * kDirectPitch + 4 * n) = make_float4(acc[4 * n], acc[4 * n + 1], acc[4 * n + 2], acc[4 * n + 3]);
  s_pix[lane] = valid ? pix : -1;
  s_tf[2 * lane] = valid ? (ho * p.Wo + wo) : 0;
  s_tf[2 * lane + 1] = utt;
  __syncwarp();
  const int sub = lane >> 3, cg = (lane & 7) * 8;
#pragma unroll 2
  for (int g = 0; g < 8; ++g) {
    const int r = g * 4 + sub;
    const long long opix = s_pix[r];
    if (opix < 0) continue;
    const float4 a0 = *reinterpret_cast<const float4*>(st + r * kDirectPitch + cg);
    const float4 a1 = *reinterpret_cast<const float4*>(st + r * kDirectPitch + cg + 4);
    const float4* b4 = reinterpret_cast<const float4*>(e.bias + (size_t)s_tf[2 * r + 1] * e.bias_stride + cg);
    float4 b0 = __ldg(b4), b1 = __ldg(b4 + 1);
    if (e.tftab) {
      const float4* t4 = reinterpret_cast<const float4*>(e.tftab + (size_t)s_tf[2 * r] * 64 + cg);
      const float4 t0 = __ldg(t4), t1 = __ldg(t4 + 1);
      b0.x += t0.x; b0.y += t0.y; b0.z += t0.z; b0.w += t0.w;
      b1.x += t1.x; b1.y += t1.y; b1.z += t1.z; b1.w += t1.w;
    }
    float v[8] = {a0.x + b0.x, a0.y + b0.y, a0.z + b0.z, a0.w + b0.w, a1.x + b1.x, a1.y + b1.y, a1.z + b1.z, a1.w + b1.w};
    if (e.relu) {
#pragma unroll
      for (int i = 0; i < 8; ++i) v[i] = fmaxf(v[i], 0.f);
    }
    uint4 o;
    o.x = pack_half2(v[0], v[1]); o.y = pack_half2(v[2], v[3]);
    o.z = pack_half2(v[4], v[5]); o.w = pack_half2(v[6], v[7]);
    *reinterpret_cast<uint4*>(e.out + opix * e.out_C + cg) = o;
  }
}

// Tensor-core version of the same convolution (legacy mma.sync path: the work is only 7 MMAC per window, but on
// CUDA cores it cost 9 % of the step).  A warp owns 16 consecutive output pixels of one image row:
// D[16 px][64 ch] = A[16 px][taps] . B[taps][64 ch] with mma.sync.m16n8k8 TF32, the A fragment gathered straight
// from the fp32 spectrogram (implicit window gather and zero padding as above).  To stay at fp32 accuracy every
// operand is split into two TF32 terms (a = a_hi + a_lo, b = b_hi + b_lo) and the three significant products are
// accumulated (3xTF32).  Kernel width must be 4 (it is, for both layers): tap k = 4 i + j.
__device__ __forceinline__ uint32_t to_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ void mma_tf32(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

constexpr int kMmaWarps = 4;
constexpr int kMmaPitch = 68;                          // floats per staged pixel row
// A warp walks one output image row (unit, ho) in 16-pixel segments, so everything that depends on the row only -
// the frame bounds, the per-utterance bias, the time-embedding row T[ho] folded into it, the output row address - is
// set up once per 13 segments; per pixel only the frequency-embedding row F[wo] (fp16, 25 KB, L1 resident) is read.
// kTab: 0 = no tables (tower), 1 = separable fp16 tables, 2 = combined fp32 table (fallback).
__device__ __forceinline__ void add_half8(float (&b)[8], const uint4 t) {
  const __half2* h = reinterpret_cast<const __half2*>(&t);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 f = __half22float2(h[i]);
    b[2 * i] += f.x;
    b[2 * i + 1] += f.y;
  }
}

template <int KSTEPS>
__global__ void __launch_bounds__(kMmaWarps * 32)     // 80 registers; capping them for 7-8 blocks/SM spills and is 15 % slower
direct_conv_mma_kernel(const DirectDev p, const int segs) {
  extern __shared__ float4 s_b[];                      // [ksteps][8 n-tiles][32 lanes] {b0_hi, b1_hi, b0_lo, b1_lo}
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* st = reinterpret_cast<float*>(s_b + KSTEPS * 8 * 32) + warp * 16 * kMmaPitch;
  for (int idx = threadIdx.x; idx < KSTEPS * 8 * 32; idx += blockDim.x) {
    const int l = idx & 31, nt = (idx >> 5) & 7, ks = idx >> 8;
    const int n = nt * 8 + (l >> 2);                   // B fragment: b0 = (k = l % 4, n), b1 = (k + 4, n)
    const float w0 = p.w[(ks * 8 + (l & 3)) * 64 + n], w1 = p.w[(ks * 8 + (l & 3) + 4) * 64 + n];
    const float h0 = __uint_as_float(to_tf32(w0)), h1 = __uint_as_float(to_tf32(w1));
    s_b[idx] = make_float4(h0, h1, __uint_as_float(to_tf32(w0 - h0)), __uint_as_float(to_tf32(w1 - h1)));
  }
  __syncthreads();
  const EpiDev& e = p.epi;
  const int rows = p.units * p.Ho;
  const int g4 = lane >> 2, t4 = lane & 3;             // fragment row / column ids
  const int sub = lane >> 3, cg = (lane & 7) * 8;      // epilogue: 4 pixels per pass, 8 channels per lane
  const int tab = (e.ttab16 && e.ftab16) ? 1 : (e.tftab ? 2 : 0);
  const int xshift = e.o_sw == 1 ? 0 : (e.o_sw == 2 ? 1 : -1);
  for (int rowid = blockIdx.x * kMmaWarps + warp; rowid < rows; rowid += gridDim.x * kMmaWarps) {
    const int unit = rowid / p.Ho, ho = rowid - unit * p.Ho;
    const int frame0 = p.units_tab.frame[unit] + p.raw_oh;
    const int lo = p.units_tab.lo[unit], hi = p.units_tab.hi[unit];
    const int utt = p.units_tab.utt ? p.units_tab.utt[unit] : 0;
    // source rows of the 2 KSTEPS kernel rows (null when the row is padding or another utterance's frame)
    const float* src[2 * KSTEPS];
#pragma unroll
    for (int i = 0; i < 2 * KSTEPS; ++i) {
      const int r = ho * p.sh + i - p.pt;
      const int frame = frame0 + r;
      src[i] = (r >= 0 && r < p.Hin && frame >= lo && frame < hi) ? e.raw + (size_t)frame * 201 : nullptr;
    }
    float bias[8];
    {
      const float4* b4 = reinterpret_cast<const float4*>(e.bias + (size_t)utt * e.bias_stride + cg);
      const float4 b0 = __ldg(b4), b1 = __ldg(b4 + 1);
      bias[0] = b0.x; bias[1] = b0.y; bias[2] = b0.z; bias[3] = b0.w;
      bias[4] = b1.x; bias[5] = b1.y; bias[6] = b1.z; bias[7] = b1.w;
      if (tab == 1) add_half8(bias, __ldg(reinterpret_cast<const uint4*>(e.ttab16 + ho * 64 + cg)));
    }
    const int yy = ho + e.o_oy;
    const long long row_pix = unit * e.o_ustride + (yy / e.o_sh) * e.o_rstride;
    const int plane_y = (yy % e.o_sh) * e.o_sw;
    for (int seg = 0; seg < segs; ++seg) {
      const int wo0 = seg * 16;
      float acc[8][4];
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) { acc[nt][0] = acc[nt][1] = acc[nt][2] = acc[nt][3] = 0.f; }
      const int f0 = (wo0 + g4) * p.sw + t4 - p.pl, f1 = f0 + 8 * p.sw;
      const bool ok0 = f0 >= 0 && f0 < p.Win, ok1 = f1 >= 0 && f1 < p.Win;
#pragma unroll
      for (int ks = 0; ks < KSTEPS; ++ks) {
        // A fragment: a0 = (px g4, tap t4), a1 = (px g4 + 8, tap t4), a2 = (px g4, tap t4 + 4), a3 = (px g4 + 8, tap t4 + 4)
        float av[4];
#pragma unroll
        for (int h = 0; h < 2; ++h) {                  // h: kernel row 2 ks + h  (taps t4 and t4 + 4)
          const float* row = src[2 * ks + h];
          av[2 * h] = (row && ok0) ? __ldg(row + f0) : 0.f;
          av[2 * h + 1] = (row && ok1) ? __ldg(row + f1) : 0.f;
        }
        uint32_t a_hi[4], a_lo[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          a_hi[k] = to_tf32(av[k]);
          a_lo[k] = to_tf32(av[k] - __uint_as_float(a_hi[k]));
        }
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
          const float4 b = s_b[(ks * 8 + nt) * 32 + lane];
          mma_tf32(acc[nt], a_lo, __float_as_uint(b.x), __float_as_uint(b.y));
          mma_tf32(acc[nt], a_hi, __float_as_uint(b.z), __float_as_uint(b.w));
          mma_tf32(acc[nt], a_hi, __float_as_uint(b.x), __float_as_uint(b.y));
        }
      }
      // C fragment -> staging: c0/c1 = (px g4, ch 8 nt + 2 t4 + {0,1}), c2/c3 = (px g4 + 8, ...)
      __syncwarp();
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        *reinterpret_cast<float2*>(st + g4 * kMmaPitch + nt * 8 + 2 * t4) = make_float2(acc[nt][0], acc[nt][1]);
        *reinterpret_cast<float2*>(st + (g4 + 8) * kMmaPitch + nt * 8 + 2 * t4) = make_float2(acc[nt][2], acc[nt][3]);
      }
      __syncwarp();
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        const int px = g * 4 + sub, wo = wo0 + px;
        if (wo >= p.Wo) continue;
        const float4 a0 = *reinterpret_cast<const float4*>(st + px * kMmaPitch + cg);
        const float4 a1 = *reinterpret_cast<const float4*>(st + px * kMmaPitch + cg + 4);
        float v[8] = {bias[0], bias[1], bias[2], bias[3], bias[4], bias[5], bias[6], bias[7]};
        if (tab == 1) {
          add_half8(v, __ldg(reinterpret_cast<const uint4*>(e.ftab16 + wo * 64 + cg)));
        } else if (tab == 2) {
          const float4* t4p = reinterpret_cast<const float4*>(e.tftab + ((size_t)ho * p.Wo + wo) * 64 + cg);
          const float4 t0 = __ldg(t4p), t1 = __ldg(t4p + 1);
          v[0] += t0.x; v[1] += t0.y; v[2] += t0.z; v[3] += t0.w;
          v[4] += t1.x; v[5] += t1.y; v[6] += t1.z; v[7] += t1.w;
        }
        v[0] += a0.x; v[1] += a0.y; v[2] += a0.z; v[3] += a0.w;
        v[4] += a1.x; v[5] += a1.y; v[6] += a1.z; v[7] += a1.w;
        if (e.relu) {
#pragma unroll
          for (int i = 0; i < 8; ++i) v[i] = fmaxf(v[i], 0.f);
        }
        const int xx = wo + e.o_ox;
        long long pix;
        if (xshift >= 0) pix = (long long)(plane_y + (xx & ((1 << xshift) - 1))) * e.o_plane + row_pix + (xx >> xshift);
        else pix = (long long)(plane_y + (xx % e.o_sw)) * e.o_plane + row_pix + (xx / e.o_sw);
        uint4 o;
        o.x = pack_half2(v[0], v[1]); o.y = pack_half2(v[2], v[3]);
        o.z = pack_half2(v[4], v[5]); o.w = pack_half2(v[6], v[7]);
        *reinterpret_cast<uint4*>(e.out + pix * e.out_C + cg) = o;
      }
    }
  }
}

// ---- first convolution per frame + window expansion (kernels.h FrameConvDev) ----
constexpr int kVirt = 17;                               // virtual frames on either side of an utterance (window half)

// grid: rows; block 256: items (w, 8-channel group).  Kernel rows i = 0..3 read frames vf - 1 + i of the
// zero-extended utterance; variants: 0 = all rows, 1 = rows 1..3 (window row 0), 2 = rows 0..2 (row 33), 3 = rows 0..1 (row 34).
__global__ void __launch_bounds__(256)
frame_conv_kernel(const FrameConvDev p) {
  __shared__ float s_w[16 * 64];
  __shared__ int s_u;
  for (int i = threadIdx.x; i < 16 * 64; i += blockDim.x) s_w[i] = p.w[i];
  const long long crow = p.crow0 + blockIdx.x;
  if (threadIdx.x == 0) {
    int a = p.u_first, b = p.u_last + 1;               // largest u with frame_offs[u] + 34 u <= crow
    while (b - a > 1) {
      const int mid = (a + b) >> 1;
      if (p.frame_offs[mid] + 2LL * kVirt * mid <= crow) a = mid; else b = mid;
    }
    s_u = a;
  }
  __syncthreads();
  const int u = s_u;
  const long long f0 = p.frame_offs[u];
  const int T = (int)(p.frame_offs[u + 1] - f0);
  const int vf = (int)(crow - (f0 + 2LL * kVirt * u)) - kVirt;    // virtual frame of this row
  const float* rows[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int fr = vf - 1 + i;
    rows[i] = (fr >= 0 && fr < T) ? p.raw + (size_t)(f0 + fr) * 201 : nullptr;
  }
  float* out = p.C + (size_t)blockIdx.x * 201 * 64;
  const size_t vplane = (size_t)p.crow_cap * 201 * 64;
  for (int it = threadIdx.x; it < 201 * 16; it += blockDim.x) {
    const int w = it >> 4, cg = (it & 15) * 4;
    float P[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
#pragma unroll
      for (int c = 0; c < 4; ++c) P[i][c] = 0.f;
      if (!rows[i]) continue;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int f = w - 1 + j;
        if (f < 0 || f >= 201) continue;
        const float x = __ldg(rows[i] + f);
        const float4 w0 = *reinterpret_cast<const float4*>(&s_w[(i * 4 + j) * 64 + cg]);
        P[i][0] = fmaf(x, w0.x, P[i][0]); P[i][1] = fmaf(x, w0.y, P[i][1]); P[i][2] = fmaf(x, w0.z, P[i][2]); P[i][3] = fmaf(x, w0.w, P[i][3]);
      }
    }
    // everything that does not depend on the window row: conditioning bias of this utterance + F[w]
    float add[4];
    {
      const float4 b0 = __ldg(reinterpret_cast<const float4*>(p.bias + (size_t)u * p.bias_stride + cg));
      add[0] = b0.x; add[1] = b0.y; add[2] = b0.z; add[3] = b0.w;
      if (p.ftab16) {
        const uint2 t = __ldg(reinterpret_cast<const uint2*>(p.ftab16 + w * 64 + cg));
        const float2 f0 = __half22float2(*reinterpret_cast<const __half2*>(&t.x)), f1 = __half22float2(*reinterpret_cast<const __half2*>(&t.y));
        add[0] += f0.x; add[1] += f0.y; add[2] += f1.x; add[3] += f1.y;
      }
    }
    float v[4][4];
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const float p01 = P[0][c] + P[1][c];
      v[3][c] = p01 + add[c];
      v[2][c] = (p01 + P[2][c]) + add[c];
      v[0][c] = ((p01 + P[2][c]) + P[3][c]) + add[c];
      v[1][c] = ((P[1][c] + P[2][c]) + P[3][c]) + add[c];
    }
#pragma unroll
    for (int k = 0; k < 4; ++k)
      *reinterpret_cast<float4*>(out + k * vplane + (size_t)w * 64 + cg) = make_float4(v[k][0], v[k][1], v[k][2], v[k][3]);
  }
}

// grid: (ceil(units / 8), ceil(Wo / CW)); a warp owns one window and walks its 35 rows over a CW-pixel column chunk,
// so the 8 warps of a CTA re-read the same C rows (row h of window n is row h - 1 of window n + 1) from L1 / L2.
template <int CW>
__global__ void __launch_bounds__(256)
window_expand_kernel(const DirectDev p, const float* __restrict__ C, long long crow0, long long crow_cap, int unit0, int unit1) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int unit = unit0 + blockIdx.x * 8 + warp;
  if (unit >= unit1) return;
  const EpiDev& e = p.epi;
  const int cg = (lane & 7) * 8;
  const int utt = p.units_tab.utt ? p.units_tab.utt[unit] : 0;
  const long long crow_n = (long long)p.units_tab.frame[unit] + 2LL * kVirt * utt - crow0;   // C row of window row 0
  const size_t vplane = (size_t)crow_cap * 201 * 64;
  constexpr int NIT = CW / 4;
  // per-lane pixel offsets of the column iterations (independent of the window row)
  long long off[NIT];
#pragma unroll
  for (int it = 0; it < NIT; ++it) {
    const int xx = blockIdx.y * CW + (lane >> 3) + 4 * it + e.o_ox;
    off[it] = ((long long)(xx % e.o_sw) * e.o_plane + unit * e.o_ustride + (xx / e.o_sw)) * e.out_C + cg;
  }
  const int wo0 = blockIdx.y * CW + (lane >> 3);
  const float* cbase = C + (size_t)crow_n * 201 * 64 + cg;
  for (int h = 0; h < p.Ho; ++h) {
    const int variant = h == 0 ? 1 : (h == p.Ho - 2 ? 2 : (h == p.Ho - 1 ? 3 : 0));
    const float* crow = cbase + variant * vplane + (size_t)h * 201 * 64;
    float bt[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (e.ttab16) add_half8(bt, __ldg(reinterpret_cast<const uint4*>(e.ttab16 + h * 64 + cg)));
    const int yy = h + e.o_oy;
    __half* orow = e.out + ((long long)((yy % e.o_sh) * e.o_sw) * e.o_plane + (long long)(yy / e.o_sh) * e.o_rstride) * e.out_C;
#pragma unroll
    for (int it = 0; it < NIT; ++it) {
      const int wo = wo0 + 4 * it;
      if (wo >= p.Wo) continue;
      const float4* c4 = reinterpret_cast<const float4*>(crow + (size_t)wo * 64);
      const float4 a0 = __ldg(c4), a1 = __ldg(c4 + 1);
      float v[8] = {a0.x + bt[0], a0.y + bt[1], a0.z + bt[2], a0.w + bt[3], a1.x + bt[4], a1.y + bt[5], a1.z + bt[6], a1.w + bt[7]};
      if (e.relu) {
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] = fmaxf(v[i], 0.f);
      }
      uint4 o;
      o.x = pack_half2(v[0], v[1]); o.y = pack_half2(v[2], v[3]);
      o.z = pack_half2(v[4], v[5]); o.w = pack_half2(v[6], v[7]);
      // streaming store: the 1.8 GB of activations must not push the per-frame table out of L2 (-9 % kernel time)
      __stcs(reinterpret_cast<uint4*>(orow + off[it]), o);
    }
  }
}

// bias_utt[u][j] = emb_a[u] . Pa[:, j] + emb_b[u] . Pb[:, j] + c[j]   (all 32 conditioning projections of
// main.py:142-148 with the batch-norm scale of their site folded in; one small fp32 GEMM per batch)
constexpr int kCondU = 8;
__global__ void __launch_bounds__(128)
cond_table_kernel(const float* __restrict__ emb_a, int stride_a, const float* __restrict__ emb_b, int stride_b, int U, const float* __restrict__ Pa,
                  const float* __restrict__ Pb, const float* __restrict__ c, int n_cols, float* __restrict__ out) {
  __shared__ float s_a[kCondU][512];
  __shared__ float s_b[kCondU][512];
  const int u0 = blockIdx.y * kCondU;
  for (int i = threadIdx.x; i < kCondU * 512; i += blockDim.x) {
    const int uu = i >> 9, k = i & 511;
    const bool ok = u0 + uu < U;
    s_a[uu][k] = ok ? emb_a[(size_t)(u0 + uu) * stride_a + k] : 0.f;
    s_b[uu][k] = ok ? emb_b[(size_t)(u0 + uu) * stride_b + k] : 0.f;
  }
  __syncthreads();
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n_cols) return;
  float acc[kCondU];
#pragma unroll
  for (int uu = 0; uu < kCondU; ++uu) acc[uu] = 0.f;
  for (int k = 0; k < 512; ++k) {
    const float pa = Pa[(size_t)k * n_cols + j], pb = Pb[(size_t)k * n_cols + j];
#pragma unroll
    for (int uu = 0; uu < kCondU; ++uu) acc[uu] = fmaf(s_a[uu][k], pa, fmaf(s_b[uu][k], pb, acc[uu]));
  }
  const float cj = c[j];
#pragma unroll
  for (int uu = 0; uu < kCondU; ++uu)
    if (u0 + uu < U) out[(size_t)(u0 + uu) * n_cols + j] = acc[uu] + cj;
}

// tf.nn.avg_pool2d over the whole 23 x 26 map (main.py:199-202): emb[n][c] = mean_p act[n][p][c]
__global__ void mean_pool_kernel(const __half* __restrict__ act, int pixels, int C, float* __restrict__ emb) {
  const int n = blockIdx.x;
  for (int c2 = threadIdx.x; c2 < C / 2; c2 += blockDim.x) {
    float sx = 0.f, sy = 0.f;
    const __half2* p = reinterpret_cast<const __half2*>(act + (size_t)n * pixels * C) + c2;
    for (int i = 0; i < pixels; ++i) {
      const float2 v = __half22float2(p[(size_t)i * (C / 2)]);
      sx += v.x; sy += v.y;
    }
    emb[(size_t)n * C + 2 * c2] = sx / (float)pixels;
    emb[(size_t)n * C + 2 * c2 + 1] = sy / (float)pixels;
  }
}

// Second stage of the split-K head (kernels.h GemmDev::ksplit): partial sums are added in split order, so the result
// does not depend on which CTA finished first.
__global__ void head_reduce_kernel(const float* __restrict__ scratch, int ksplit, int units, int N, const float* __restrict__ scale,
                                   const float* __restrict__ bias, const float* __restrict__ raw, const int* __restrict__ frame,
                                   float* __restrict__ out) {
  const int n = blockIdx.x;
  const size_t plane = (size_t)units * N;
  const float* raw_row = raw + (size_t)frame[n] * 201;
  for (int c = threadIdx.x; c < 201; c += blockDim.x) {
    float acc = 0.f;
    for (int s = 0; s < ksplit; ++s) acc += scratch[s * plane + (size_t)n * N + c];
    out[(size_t)n * 201 + c] = acc * scale[c] + bias[c] + raw_row[c];
  }
}

// Window n of the chunk is global frame w0 + n (one window per STFT frame, SN/apply.py:378); its clip is
// found by binary search in frame_offs.
__global__ void units_main_kernel(const long long* __restrict__ frame_offs, int U, int w0, int nwin, int* frame, int* lo,
                                  int* hi, int* utt) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= nwin) return;
  const long long g = (long long)w0 + n;
  int a = 0, b = U;                                     // frame_offs[a] <= g < frame_offs[b]
  while (b - a > 1) {
    const int mid = (a + b) >> 1;
    if (frame_offs[mid] <= g) a = mid; else b = mid;
  }
  frame[n] = (int)g;
  lo[n] = (int)frame_offs[a];
  hi[n] = (int)frame_offs[a + 1];
  utt[n] = a;
}

__global__ void units_rows_kernel(int r0, int n_units, int rows, int* frame, int* lo, int* hi, int* utt) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= n_units) return;
  frame[n] = (r0 + n) * rows;
  lo[n] = (r0 + n) * rows;
  hi[n] = (r0 + n + 1) * rows;
  utt[n] = 0;
}

}  // namespace

cudaError_t launch_direct_conv(cudaStream_t s, const DirectDev& p) {
  if (p.units <= 0) return cudaSuccess;
  if (p.N != 64) return cudaErrorInvalidValue;
  if (p.kw == 4 && p.kh == 4) {
    const int segs = (p.Wo + 15) / 16;
    const long long rows = (long long)p.units * p.Ho;
    if (rows > 0x7fffffffLL) return cudaErrorInvalidValue;
    const size_t smem_mma = (size_t)2 * 8 * 32 * 16 + kMmaWarps * 16 * kMmaPitch * 4;
    long long blocks_mma = (rows + kMmaWarps - 1) / kMmaWarps;
    if (blocks_mma > 148 * 16) blocks_mma = 148 * 16;              // grid-stride: the weight fragments are staged once per CTA
    direct_conv_mma_kernel<2><<<(unsigned)blocks_mma, kMmaWarps * 32, smem_mma, s>>>(p, segs);
    return cudaGetLastError();
  }
  const long long total = (long long)p.units * p.Ho * p.Wo;
  const int threads = 128;
  const long long blocks = (total + threads - 1) / threads;
  const size_t smem = (size_t)p.kh * p.kw * 64 * 4 + 4 * 32 * kDirectPitch * 4 + 2 * 4 * 32 * 4 + 4 * 64 * 4;
  direct_conv64_kernel<<<(unsigned)blocks, threads, smem, s>>>(p);
  return cudaGetLastError();
}

cudaError_t launch_frame_conv(cudaStream_t s, const FrameConvDev& p) {
  if (p.rows <= 0) return cudaSuccess;
  frame_conv_kernel<<<p.rows, 256, 0, s>>>(p);
  return cudaGetLastError();
}

cudaError_t launch_window_expand(cudaStream_t s, const DirectDev& d, const float* C, long long crow0, long long crow_cap, int unit0,
                                 int unit1) {
  if (unit1 <= unit0) return cudaSuccess;
  if (d.N != 64 || d.kh != 4 || d.kw != 4 || d.sh != 1 || d.sw != 1 || d.pt != 1 || d.pl != 1 || d.Win != 201) return cudaErrorInvalidValue;
  window_expand_kernel<8><<<dim3((unit1 - unit0 + 7) / 8, (d.Wo + 7) / 8), 256, 0, s>>>(d, C, crow0, crow_cap, unit0, unit1);
  return cudaGetLastError();
}

cudaError_t launch_cond_table(cudaStream_t s, const float* emb_a, int stride_a, const float* emb_b, int stride_b, int U, const float* Pa,
                              const float* Pb, const float* c, int n_cols, float* out) {
  if (U <= 0) return cudaSuccess;
  dim3 grid((n_cols + 127) / 128, (U + kCondU - 1) / kCondU);
  cond_table_kernel<<<grid, 128, 0, s>>>(emb_a, stride_a, emb_b, stride_b, U, Pa, Pb, c, n_cols, out);
  return cudaGetLastError();
}

cudaError_t launch_mean_pool(cudaStream_t s, const __half* act, int units, int pixels, int C, float* emb) {
  if (units <= 0) return cudaSuccess;
  mean_pool_kernel<<<units, 256, 0, s>>>(act, pixels, C, emb);
  return cudaGetLastError();
}

cudaError_t launch_head_reduce(cudaStream_t s, const float* scratch, int ksplit, int units, int N, const float* scale, const float* bias,
                               const float* raw, const int* frame, float* out) {
  if (units <= 0) return cudaSuccess;
  head_reduce_kernel<<<units, 224, 0, s>>>(scratch, ksplit, units, N, scale, bias, raw, frame, out);
  return cudaGetLastError();
}

cudaError_t launch_units_main(cudaStream_t s, const long long* frame_offs, int U, int w0, int nwin, int* frame, int* lo,
                              int* hi, int* utt) {
  if (nwin <= 0) return cudaSuccess;
  units_main_kernel<<<(nwin + 255) / 256, 256, 0, s>>>(frame_offs, U, w0, nwin, frame, lo, hi, utt);
  return cudaGetLastError();
}

cudaError_t launch_units_rows(cudaStream_t s, int r0, int n, int rows_per_unit, int* frame, int* lo, int* hi, int* utt) {
  if (n <= 0) return cudaSuccess;
  units_rows_kernel<<<(n + 255) / 256, 256, 0, s>>>(r0, n, rows_per_unit, frame, lo, hi, utt);
  return cudaGetLastError();
}

}  // namespace nhans
