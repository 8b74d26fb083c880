// Row-walk convolution on the 5th-generation tensor cores (sm_100a): the 64-channel stride-1 4 x 4 layers of the
// mask network (resblock1_1_conv2, resblock1_2_conv1 / conv2; N_HANS___Selective_Noise/main.py:162-186, 221-222).
//
// Why a second tensor-core kernel.  As a GEMM these layers have N = 64, and an M = 128 tcgen05.mma with N = 64 is
// bound by its shared-memory operand reads (4 KB of A per 32 cycles).  Round 1 paired pixels to reach N = 128,
// which costs 20 % zero weight blocks and still re-reads every activation row from L2 once per kernel row
// (57 % of the tensor peak, a third of the whole step).  Here the roles are turned around: a CTA owns a strip of
// 128 pixels (unit, x) and WALKS DOWN the 35 image rows of the strip.  Input row r is loaded once (one TMA slab,
// the four column taps read it through row-shifted UMMA descriptors) and multiplied by the weights of all four
// kernel rows at once: B block bi = kernel row 3 - bi, so one N = 256 MMA accumulates into the four output rows
// r - 2 .. r + 1 that see input row r.  Output rows live in a ring of 8 TMEM slots of 64 columns (all 512
// columns); a slot is claimed when its output row gets its first input row, published to the epilogue after its
// last one, and freed when the epilogue has read it.  Every MMA is dense (no zero blocks, no margin rows), the
// weights (4 x 32 KB) stay resident in shared memory for the whole launch, A comes from L2 once per layer instead
// of four times, and the MMAs run at N = 256 except where the ring wraps or a fresh slot must not accumulate
// (walk_sched.h; checked on the host by tests/host/walk_sched_check.cc).
//
//   warp 8      producer: the resident weights once, then one A slab per (tile, input row)
//   warps 10-15 (resblock1_1_conv2 only) build the A slabs themselves from the per-frame table of the first
//               convolution - relu(C[variant][frame + row][x] + T1[row]) -> fp16, written with TMA's 128-byte swizzle -
//               so the first activation tensor (1.8 GB written + read per 2048-window pass) never exists in HBM
//   warp 9      MMA issuer: 16 K steps (4 column taps x 4 x K = 16) per input row over the sliding slot window
//   warps 0-7   epilogue, row per thread (thread = TMEM lane = pixel): everything that does not depend on the
//               image row - the conditioning bias of the pixel's utterance and the frequency embedding F[x] - is
//               held in registers for the whole strip; per output row: T[h] from shared memory, the identity
//               residual (256-bit loads, prefetched one row ahead) or the rank-1 transform term, ReLU, 256-bit
//               fp16 stores into the consumer's grid.
#include <cstdio>
#include <cstdlib>

#include "kernels.h"
#include "ptx.cuh"
#include "walk_sched.h"

namespace nhans {

namespace {

constexpr int kSlabBytes = kSlabRows * 128;
constexpr int kNA = 4;                             // A slab ring
constexpr int kBTile = 64 * kWalkKH * 128;         // one column tap: [4 kernel rows x 64 couts] x 64 cin, fp16
constexpr int kBBytes = kWalkKW * kBTile;          // 128 KB resident
constexpr int kCtrlBytes = 1024;
constexpr int kMaxH = 40;
constexpr int kTabBytes = kMaxH * 64 * 4 + 2 * 64 * 4;
constexpr int kWalkThreads = 320;                  // 8 epilogue warps + producer + MMA issuer
constexpr int kGenWarps = 6;                       // + slab generator warps (kWalkGen launches only; 512 threads x 128 registers)
constexpr int kWarpA = 8, kWarpMma = 9, kWarpGen0 = 10;
constexpr int kWalkSmem = 1024 + kNA * kSlabBytes + kBBytes + kCtrlBytes + kTabBytes;
static_assert(kWalkSmem <= 227 * 1024, "shared memory budget");

constexpr int kWalkRes = 1;                        // + res_scale[c] * x (identity residual)
constexpr int kWalkR1 = 2;                         // + r1_vec[c] * raw spectrogram value (1x1 transform with Cin = 1)
constexpr int kWalkGen = 4;                        // A slabs generated from the per-frame table of the first convolution

struct __align__(8) WalkCtrl {
  uint64_t a_full[kNA], a_empty[kNA];
  uint64_t b_full;
  uint64_t tmem_full[kWalkSlots], tmem_empty[kWalkSlots];
  uint32_t tmem_base;
  uint32_t pad;
};
static_assert(sizeof(WalkCtrl) <= kCtrlBytes, "control block too large");

template <int EPI>
__global__ void __launch_bounds__(kWalkThreads + ((EPI & 4) ? kGenWarps * 32 : 0), 1)
conv64_walk_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB, const WalkDev p) {
  constexpr bool kRes = (EPI & kWalkRes) != 0, kR1 = (EPI & kWalkR1) != 0, kGen = (EPI & kWalkGen) != 0;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = ptx::smem_u32(smem_raw);
  uint8_t* smem = smem_raw + ((1024u - (raw_addr & 1023u)) & 1023u);
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + kNA * kSlabBytes;
  WalkCtrl* ctrl = reinterpret_cast<WalkCtrl*>(smem_b + kBBytes);
  float* s_t = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(ctrl) + kCtrlBytes);    // [H][64] time embedding, fp32
  float* s_rs = s_t + kMaxH * 64;                                                          // [64] residual scale
  float* s_r1 = s_rs + 64;                                                                 // [64] rank-1 vector

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int H = p.H;
  const int num_tiles = (p.plane_rows + 127) >> 7;
  const EpiDev& e = p.epi;

  for (int i = threadIdx.x; i < H * 64; i += blockDim.x) s_t[i] = e.ttab16 ? __half2float(e.ttab16[i]) : 0.f;
  if (threadIdx.x < 64) {
    s_rs[threadIdx.x] = kRes ? e.res_scale[threadIdx.x] : 0.f;
    s_r1[threadIdx.x] = kR1 ? e.r1_vec[threadIdx.x] : 0.f;
  }
  if (threadIdx.x == 0) {
    // a_full: one TMA transaction arrival, or one arrival per generator warp
    for (int s = 0; s < kNA; ++s) { ptx::mbar_init(&ctrl->a_full[s], kGen ? kGenWarps : 1); ptx::mbar_init(&ctrl->a_empty[s], 1); }
    ptx::mbar_init(&ctrl->b_full, 1);
    for (int s = 0; s < kWalkSlots; ++s) { ptx::mbar_init(&ctrl->tmem_full[s], 1); ptx::mbar_init(&ctrl->tmem_empty[s], 8); }
    ptx::fence_barrier_init();
    ptx::fence_proxy_async();
  }
  if (warp == kWarpA && lane == 0) {
    ptx::tma_prefetch_desc(&mapA);
    ptx::tma_prefetch_desc(&mapB);
  }
  if (warp == kWarpMma) ptx::tmem_alloc(&ctrl->tmem_base, 512);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = ctrl->tmem_base;

  if (warp == kWarpA) {
    // ===================== producer: resident weights, then one A slab per (tile, input row) =====================
    if (ptx::elect_one()) {
      ptx::mbar_expect_tx(&ctrl->b_full, (uint32_t)kBBytes);
      for (int kw = 0; kw < kWalkKW; ++kw) ptx::tma_load_2d(smem_b + (size_t)kw * kBTile, &mapB, &ctrl->b_full, kw * 64, 0);
    }
    __syncwarp();
    uint32_t slot = 0, phase = 0;
    if (!kGen) {
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        const int m0 = tile * 128 - p.pl;
        for (int r = 0; r < H; ++r) {
          ptx::mbar_wait(&ctrl->a_empty[slot], phase ^ 1, p.err_flag, 1);
          if (ptx::elect_one()) {
            ptx::mbar_expect_tx(&ctrl->a_full[slot], (uint32_t)kSlabBytes);
            ptx::tma_load_2d(smem_a + (size_t)slot * kSlabBytes, &mapA, &ctrl->a_full[slot], 0, r * p.plane_pitch + m0);
          }
          __syncwarp();
          if (++slot == (uint32_t)kNA) { slot = 0; phase ^= 1; }
        }
      }
    }
  } else if (kGen && warp >= kWarpGen0) {
    // ===================== slab generators (6 warps): the first convolution's output never goes to HBM =====================
    // Slab row j is pixel m0 + j = (unit, x); a lane owns one 16-byte chunk (8 channels) of one row per iteration and
    // writes it where TMA's 128-byte swizzle would have put it: chunk c of row j at j * 128 + ((c ^ (j & 7)) << 4).
    // All table loads of a step are issued before the wait for the free slab, so L2 latency overlaps the MMAs.
    constexpr int kIts = (kSlabRows + 4 * kGenWarps - 1) / (4 * kGenWarps);   // rows per lane
    const int gw = warp - kWarpGen0;
    const int c8 = lane & 7, cg = c8 * 8;
    const size_t vplane = (size_t)p.gen_crow_cap * 201 * 64;
    const int n_units = p.plane_rows / p.Wq;
    uint32_t slot = 0, phase = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
      const int m0 = tile * 128 - p.pl;
      // the 136 rows span at most two units
      const int unitA = (m0 < 0 ? 0 : m0) / p.Wq;
      const int xA = m0 - unitA * p.Wq;                                     // x of slab row 0 relative to unit A (may be -1)
      long long crowA = -1, crowB = -1;
      if (unitA < n_units) crowA = (long long)p.units.frame[unitA] + (long long)kWinReach * p.units.utt[unitA] - p.gen_crow0;
      if (unitA + 1 < n_units) crowB = (long long)p.units.frame[unitA + 1] + (long long)kWinReach * p.units.utt[unitA + 1] - p.gen_crow0;
      // per-lane source offsets of its rows (independent of the image row): -1 = zero row (margin / outside the pass)
      long long src_off[kIts];
#pragma unroll
      for (int it = 0; it < kIts; ++it) {
        const int j = it * (4 * kGenWarps) + gw * 4 + (lane >> 3);
        int x = xA + j;
        long long crow = crowA;
        if (x >= p.Wq) { x -= p.Wq; crow = crowB; }
        src_off[it] = (j < kSlabRows && x >= 0 && x < p.Wo && crow >= 0) ? (crow * 201 + x) * 64 + cg : -1;
      }
      for (int r = 0; r < H; ++r) {
        const int variant = r == 0 ? 1 : (r == H - 2 ? 2 : (r == H - 1 ? 3 : 0));
        const float* plane = p.gen_C + (size_t)variant * vplane + (size_t)r * 201 * 64;
        float4 va[kIts], vb[kIts];
#pragma unroll
        for (int it = 0; it < kIts; ++it) {
          if (src_off[it] >= 0) {
            const float4* src = reinterpret_cast<const float4*>(plane + src_off[it]);
            va[it] = __ldg(src);
            vb[it] = __ldg(src + 1);
          }
        }
        float t8[8];
        {
          const uint4 tv = __ldg(reinterpret_cast<const uint4*>(p.gen_ttab16 + r * 64 + cg));
          const __half2* th = reinterpret_cast<const __half2*>(&tv);
#pragma unroll
          for (int k = 0; k < 4; ++k) { const float2 f = __half22float2(th[k]); t8[2 * k] = f.x; t8[2 * k + 1] = f.y; }
        }
        ptx::mbar_wait(&ctrl->a_empty[slot], phase ^ 1, p.err_flag, 1);
        uint8_t* slab = smem_a + (size_t)slot * kSlabBytes;
#pragma unroll
        for (int it = 0; it < kIts; ++it) {
          const int j = it * (4 * kGenWarps) + gw * 4 + (lane >> 3);
          if (j >= kSlabRows) continue;
          uint4 o = make_uint4(0u, 0u, 0u, 0u);
          if (src_off[it] >= 0) {
            const float4 a = va[it], b = vb[it];
            o.x = ptx::pack_half2(fmaxf(a.x + t8[0], 0.f), fmaxf(a.y + t8[1], 0.f));
            o.y = ptx::pack_half2(fmaxf(a.z + t8[2], 0.f), fmaxf(a.w + t8[3], 0.f));
            o.z = ptx::pack_half2(fmaxf(b.x + t8[4], 0.f), fmaxf(b.y + t8[5], 0.f));
            o.w = ptx::pack_half2(fmaxf(b.z + t8[6], 0.f), fmaxf(b.w + t8[7], 0.f));
          }
          *reinterpret_cast<uint4*>(slab + j * 128 + ((c8 ^ (j & 7)) << 4)) = o;
        }
        ptx::fence_proxy_async();                // generic-proxy writes -> visible to the tensor core's async-proxy reads
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(&ctrl->a_full[slot]);
        if (++slot == (uint32_t)kNA) { slot = 0; phase ^= 1; }
      }
    }
  } else if (warp >= kWarpGen0) {
    // no generated operand: the two extra warps have nothing to do
  } else if (warp == kWarpMma) {
    // ===================== MMA issuer =====================
    const uint32_t idesc0 = (1u << 4) | ((128u >> 4) << 24);                 // fp16 x fp16 -> fp32, M = 128; N added per segment
    const uint64_t desc_hi = ptx::umma_desc_sw128(0, 0);
    const uint32_t a_base = ptx::smem_u32(smem_a) >> 4, b_base = ptx::smem_u32(smem_b) >> 4;
    long long w_a = 0, w_tmem = 0;
    const long long t_start = clock64();
    ptx::mbar_wait(&ctrl->b_full, 0, p.err_flag, 6);
    ptx::tc_fence_after();
    uint32_t aslot = 0, aphase = 0;
    long long seq = 0;
    // barrier waits of one step: the slots it claims must have been read by the epilogue, its slab must have landed
    auto wait_step = [&](long long sq, int r, uint32_t slot, uint32_t phase) {
      const WalkWin w = walk_window(sq, r, H, p.pt);
      for (int c = 0; c < w.n_fresh; ++c) {
        const long long J = sq * H + w.o_lo + w.n - w.n_fresh + c;
        ptx::mbar_wait_timed(&ctrl->tmem_empty[J & (kWalkSlots - 1)], (uint32_t)(((J >> 3) & 1) ^ 1), p.err_flag, 2, &w_tmem);
      }
      ptx::mbar_wait_timed(&ctrl->a_full[slot], phase, p.err_flag, 3, &w_a);
    };
    // (not with the generated operand: its slabs arrive just in time, and a wait in the middle of a step would hold back
    // that step's last MMAs and commits - measured 1063 vs 1095 TFLOP/s on the same box)
    if (!kGen && (int)blockIdx.x < num_tiles) wait_step(0, 0, 0, 0);
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++seq) {
      const long long j0 = seq * H;
      for (int r = 0; r < H; ++r) {
        const WalkWin w = walk_window(seq, r, H, p.pt);
        if (kGen) wait_step(seq, r, aslot, aphase);
        ptx::tc_fence_after();
        const uint32_t a_lo = a_base + aslot * (kSlabBytes >> 4);
        const uint64_t da0 = desc_hi | (uint64_t)a_lo;
        const uint64_t db0 = desc_hi | (uint64_t)b_base;
        const uint32_t d_a = tmem_base + (uint32_t)w.slot0 * 64, d_b = tmem_base;
        const uint32_t i_a = idesc0 | ((uint32_t)(w.n1 * 64 >> 3) << 17), i_b = idesc0 | ((uint32_t)((w.n - w.n1) * 64 >> 3) << 17);
        const uint64_t db_a = db0 + (uint64_t)(w.bi0 * ((64 * 128) >> 4)), db_b = db_a + (uint64_t)(w.n1 * ((64 * 128) >> 4));
        // K steps kk = 4 kw + k (tap kw = slab rows shifted by kw): one MMA over the whole window, two where the ring wraps
        auto issue = [&](int kk_lo, int kk_hi) {
          if (w.n == w.n1) {
#pragma unroll
            for (int kk = kk_lo; kk < kk_hi; ++kk) {
              const int kw = kk >> 2, k = kk & 3;
              ptx::umma_f16(d_a, da0 + (uint64_t)(kw * 8 + 2 * k), db_a + (uint64_t)(kw * (kBTile >> 4) + 2 * k), i_a, 1u);
            }
          } else {
#pragma unroll
            for (int kk = kk_lo; kk < kk_hi; ++kk) {
              const int kw = kk >> 2, k = kk & 3;
              const uint64_t da = da0 + (uint64_t)(kw * 8 + 2 * k);
              const uint64_t bo = (uint64_t)(kw * (kBTile >> 4) + 2 * k);
              ptx::umma_f16(d_a, da, db_a + bo, i_a, 1u);
              ptx::umma_f16(d_b, da, db_b + bo, i_b, 1u);
            }
          }
        };
        // one elected lane issues the whole step: K step 0 apart, because fresh slots must not accumulate
        if (ptx::elect_one()) {
          walk_segments(w, true, [&](int slot, int bi, int nb, int fresh) {
            ptx::umma_f16(tmem_base + (uint32_t)slot * 64, da0, db0 + (uint64_t)(bi * ((64 * 128) >> 4)),
                          idesc0 | ((uint32_t)(nb * 64 >> 3) << 17), fresh ? 0u : 1u);
          });
          issue(1, 12);
        }
        __syncwarp();
        // while those 12 MMAs are queued: the barrier waits of the NEXT step (an already-complete mbarrier.try_wait still
        // costs ~90 cycles, and the tensor pipe's queue is too short to cover two of them plus the window arithmetic)
        uint32_t nslot = aslot + 1, nphase = aphase;
        if (nslot == (uint32_t)kNA) { nslot = 0; nphase ^= 1; }
        if (!kGen) {
          if (r + 1 < H) wait_step(seq, r + 1, nslot, nphase);
          else if (tile + (int)gridDim.x < num_tiles) wait_step(seq + 1, 0, nslot, nphase);
        }
        if (ptx::elect_one()) {
          issue(12, kWalkKW * 4);
          ptx::umma_commit(&ctrl->a_empty[aslot]);
          for (int d = 0; d < w.n_done; ++d) ptx::umma_commit(&ctrl->tmem_full[(j0 + w.done_lo + d) & (kWalkSlots - 1)]);
        }
        __syncwarp();
        aslot = nslot; aphase = nphase;
      }
    }
    if (p.debug_stats && lane == 0) {
      atomicAdd(p.debug_stats + 0, (unsigned long long)w_tmem);
      atomicAdd(p.debug_stats + 1, (unsigned long long)w_a);
      atomicAdd(p.debug_stats + 4, (unsigned long long)(clock64() - t_start));
    }
  } else {
    // ===================== epilogue (warps 0..7) =====================
    const int q = warp & 3, half = warp >> 2;      // TMEM lane quarter; channel chunks [16 half, +16) and [32 + 16 half, +16)
    const int ch0 = half * 16;
    long long w_full = 0;
    long long seq = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++seq) {
      const long long j0 = seq * H;
      const int m_plane = tile * 128 + q * 32 + lane;
      const int unit = m_plane / p.Wq;
      const int wb = m_plane - unit * p.Wq;
      const bool ok = m_plane < p.plane_rows && wb < p.Wo;
      // everything that does not depend on the image row: conditioning bias of the utterance + F[x]
      float bf[2][16];
      int frame0 = 0, f_lo = 0, f_hi = 0;
      long long base_pix = 0;
      int xplane = 0;
      if (ok) {
        const int utt = p.units.utt ? p.units.utt[unit] : 0;
        const float* bp = e.bias + (size_t)utt * e.bias_stride;
#pragma unroll
        for (int ci = 0; ci < 2; ++ci) {
          const float4* b4 = reinterpret_cast<const float4*>(bp + ch0 + 32 * ci);
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const float4 v = __ldg(b4 + k);
            bf[ci][4 * k] = v.x; bf[ci][4 * k + 1] = v.y; bf[ci][4 * k + 2] = v.z; bf[ci][4 * k + 3] = v.w;
          }
          if (e.ftab16) {
            uint4 f0, f1;
            ptx::ldg256(e.ftab16 + (size_t)wb * 64 + ch0 + 32 * ci, f0, f1);
            const uint4 ff[2] = {f0, f1};
            const __half2* fh = reinterpret_cast<const __half2*>(ff);
#pragma unroll
            for (int k = 0; k < 8; ++k) {
              const float2 v = __half22float2(fh[k]);
              bf[ci][2 * k] += v.x;
              bf[ci][2 * k + 1] += v.y;
            }
          }
        }
        if (kR1) {
          frame0 = p.units.frame[unit] + e.raw_oh;
          f_lo = p.units.lo[unit];
          f_hi = p.units.hi[unit];
        }
        const int xx = wb + e.o_ox;
        xplane = xx % e.o_sw;
        base_pix = (long long)unit * e.o_ustride + xx / e.o_sw;
      } else {
#pragma unroll
        for (int ci = 0; ci < 2; ++ci)
#pragma unroll
          for (int k = 0; k < 16; ++k) bf[ci][k] = 0.f;
      }
      // loads of output row o that do not depend on the accumulator: issued one row ahead
      uint4 xn[2][2];
      float rawn = 0.f;
      auto issue_loads = [&](int o) {
        if (!ok || o >= H) return;
        if (kRes) {
          const __half* rp = e.res + ((size_t)o * p.plane_pitch + m_plane) * e.res_C + ch0;
          ptx::ldg256(rp, xn[0][0], xn[0][1]);
          ptx::ldg256(rp + 32, xn[1][0], xn[1][1]);
        }
        if (kR1) {
          const int frame = frame0 + o * e.r1_sh;
          rawn = (frame >= f_lo && frame < f_hi) ? __ldg(e.raw + (size_t)frame * 201 + wb * e.r1_sw) : 0.f;
        }
      };
      issue_loads(0);
#pragma unroll 1
      for (int o = 0; o < H; ++o) {
        const long long J = j0 + o;
        const uint32_t slot = (uint32_t)(J & (kWalkSlots - 1));
        uint4 xc[2][2];
        float rawv = 0.f;
        if (kRes) { xc[0][0] = xn[0][0]; xc[0][1] = xn[0][1]; xc[1][0] = xn[1][0]; xc[1][1] = xn[1][1]; }
        if (kR1) rawv = rawn;
        issue_loads(o + 1);
        ptx::mbar_wait_timed(&ctrl->tmem_full[slot], (uint32_t)((J >> 3) & 1), p.err_flag, 4, &w_full);
        ptx::tc_fence_after();
        uint32_t tv[2][16];
        const uint32_t t_addr = tmem_base + ((uint32_t)(q * 32) << 16) + slot * 64 + ch0;
        ptx::tmem_ld16(t_addr, tv[0]);
        ptx::tmem_ld16(t_addr + 32, tv[1]);
        ptx::tmem_ld_wait();
        // the accumulator slot is free as soon as it is in registers
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(&ctrl->tmem_empty[slot]);
        if (ok) {
          const int y = o + e.o_oy;
          const long long pix = (long long)((y % e.o_sh) * e.o_sw + xplane) * e.o_plane + (long long)(y / e.o_sh) * e.o_rstride + base_pix;
          __half* op = e.out + pix * e.out_C + ch0;
#pragma unroll
          for (int ci = 0; ci < 2; ++ci) {
            float f[16];
            const float4* t4 = reinterpret_cast<const float4*>(s_t + o * 64 + ch0 + 32 * ci);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const float4 t = t4[k];
              f[4 * k] = __uint_as_float(tv[ci][4 * k]) + (bf[ci][4 * k] + t.x);
              f[4 * k + 1] = __uint_as_float(tv[ci][4 * k + 1]) + (bf[ci][4 * k + 1] + t.y);
              f[4 * k + 2] = __uint_as_float(tv[ci][4 * k + 2]) + (bf[ci][4 * k + 2] + t.z);
              f[4 * k + 3] = __uint_as_float(tv[ci][4 * k + 3]) + (bf[ci][4 * k + 3] + t.w);
            }
            if (kRes) {
              const __half2* xh = reinterpret_cast<const __half2*>(xc[ci]);
              const float4* rs4 = reinterpret_cast<const float4*>(s_rs + ch0 + 32 * ci);
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                const float4 rs = rs4[k];
                const float2 x0 = __half22float2(xh[2 * k]), x1 = __half22float2(xh[2 * k + 1]);
                f[4 * k] = fmaf(rs.x, x0.x, f[4 * k]); f[4 * k + 1] = fmaf(rs.y, x0.y, f[4 * k + 1]);
                f[4 * k + 2] = fmaf(rs.z, x1.x, f[4 * k + 2]); f[4 * k + 3] = fmaf(rs.w, x1.y, f[4 * k + 3]);
              }
            }
            if (kR1) {
              const float4* r14 = reinterpret_cast<const float4*>(s_r1 + ch0 + 32 * ci);
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                const float4 r1 = r14[k];
                f[4 * k] = fmaf(r1.x, rawv, f[4 * k]); f[4 * k + 1] = fmaf(r1.y, rawv, f[4 * k + 1]);
                f[4 * k + 2] = fmaf(r1.z, rawv, f[4 * k + 2]); f[4 * k + 3] = fmaf(r1.w, rawv, f[4 * k + 3]);
              }
            }
            if (e.relu) {
#pragma unroll
              for (int k = 0; k < 16; ++k) f[k] = fmaxf(f[k], 0.f);
            }
            uint4 o0, o1;
            o0.x = ptx::pack_half2(f[0], f[1]); o0.y = ptx::pack_half2(f[2], f[3]); o0.z = ptx::pack_half2(f[4], f[5]); o0.w = ptx::pack_half2(f[6], f[7]);
            o1.x = ptx::pack_half2(f[8], f[9]); o1.y = ptx::pack_half2(f[10], f[11]); o1.z = ptx::pack_half2(f[12], f[13]); o1.w = ptx::pack_half2(f[14], f[15]);
            ptx::stg256(op + 32 * ci, o0, o1);
          }
        }
      }
    }
    if (p.debug_stats && warp == 0 && lane == 0) atomicAdd(p.debug_stats + 3, (unsigned long long)w_full);
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == kWarpMma) {
    __syncwarp();
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, 512);
  }
}

template <int EPI>
cudaError_t launch_flavour(cudaStream_t s, int grid, const CUtensorMap& a, const CUtensorMap& b, const WalkDev& p) {
  cudaError_t e = cudaFuncSetAttribute(conv64_walk_kernel<EPI>, cudaFuncAttributeMaxDynamicSharedMemorySize, kWalkSmem);
  if (e != cudaSuccess) return e;
  conv64_walk_kernel<EPI><<<grid, kWalkThreads + ((EPI & kWalkGen) ? kGenWarps * 32 : 0), kWalkSmem, s>>>(a, b, p);
  return cudaGetLastError();
}

}  // namespace

cudaError_t launch_walk(cudaStream_t s, int n_sm, const CUtensorMap& mapA, const CUtensorMap& mapB, const WalkDev& p) {
  if (p.plane_rows <= 0) return cudaSuccess;
  const EpiDev& e = p.epi;
  if (p.H < 1 || p.H > kMaxH || p.pt < 0 || p.pt > kWalkKH - 1 || e.head || e.o_mode != 0 || e.out_C != 64 ||
      (e.res && e.res_C != 64) || (e.res && e.r1_vec))
    return cudaErrorInvalidValue;
  const int tiles = (p.plane_rows + 127) / 128;
  const int grid = tiles < n_sm ? tiles : n_sm;
  if (p.gen_C) {
    // generated A operand: the layer after the first convolution (rank-1 transform epilogue, 'SAME' 4 x 4 geometry)
    if (!e.r1_vec || e.res || !p.gen_ttab16 || p.pl != 1 || p.Wo != 201) return cudaErrorInvalidValue;
    return launch_flavour<kWalkR1 | kWalkGen>(s, grid, mapA, mapB, p);
  }
  if (e.res) return launch_flavour<kWalkRes>(s, grid, mapA, mapB, p);
  if (e.r1_vec) return launch_flavour<kWalkR1>(s, grid, mapA, mapB, p);
  return launch_flavour<0>(s, grid, mapA, mapB, p);
}

}  // namespace nhans
