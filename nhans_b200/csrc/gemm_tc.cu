// Shifted-row implicit-GEMM convolution on the 5th-generation tensor cores (sm_100a).
//
//   D[m, n] = sum_g sum_{t < ntaps_g}  A_{map_g}[m + row_off_g + shift_{g,t}, col_g : col_g + 64] . B[n, 64 bk_{g,t} : +64]
//
// Every convolution and dense layer of N_HANS___Selective_Noise/main.py:98-242 except the two Cin = 1
// convolutions is lowered to this form by plan.cc (a group g = the kw taps of one kernel row and one
// 64-channel chunk).  Activations live in "image-row-outer" padded grids (plan.h): a tap is a constant row
// offset, vertical padding is TMA out-of-bounds fill, and only real output rows are enumerated; tiles are
// ordered image-row-fastest.  A tile lies in one output row ho and runs only the groups whose kernel row reads
// inside the image for that row (GemmDev::row_groups, at most two index ranges looked up once per tile): all three
// roles skip the same groups, with no test per group.  Persistent CTA PAIRS (cluster of 2, cta_group::2; a
// single-CTA instantiation serves small problems); a tile is (256 / BN) sub-tiles of 256 rows (128 per CTA) x BN
// columns, i.e. always 256 fp32 accumulator columns in TMEM, double buffered (2 x 256 = all 512 columns).
//
//   warp 8   A producer     one TMA box of 136 rows x 64 channels ("slab") per (group, sub-tile): the kw taps
//                           of a kernel row read the SAME slab through UMMA descriptors whose start address
//                           is shifted by `shift` rows, so A comes from L2 once per kernel row, not per tap;
//                           the slabs of a group complete on ONE mbarrier (ring of 4, or 6 for BN <= 128)
//   warp 9   B producer     one TMA box (BN / 2) x 64 per k-block: each CTA of a pair loads half of B; the
//                           transactions of both CTAs are credited to the leader's mbarrier, all tiles of a
//                           group to the barrier of the group's first slot
//   warp 10  MMA issuer     leader CTA only, ONE elected lane for the whole role (waits, MMAs, commits: two
//                           barrier waits per group): tcgen05.mma.cta_group::2.kind::f16, M = 256, N = BN,
//                           4 x (K = 16) per tap, two sub-tiles interleaved; tcgen05.commit...multicast
//                           releases ring slots / publishes accumulators in both CTAs; split-K for the head
//   warps 0-7 epilogue      two flavours (kEpiRow): row-per-thread for BN <= 128 (thread = TMEM lane = GEMM
//                           row, 16 channels per step, 256-bit residual loads and stores, fp16 tables and
//                           per-channel vectors in shared memory, no staging) and transposing for BN = 256 and
//                           the head (tcgen05.ld -> XOR-swizzled fp32 transpose -> 4 lanes per row, coalesced).
//                           + per-utterance conditioning bias + time / frequency embedding tables + scaled
//                           identity residual / rank-1 transform -> ReLU -> fp16 into the consumer's grid
//                           (or, for the head, raw fp32 partial sums of one K split: head_reduce_kernel
//                           adds the splits, the column scale, the bias and the centre frame)
//
// The 64-channel stride-1 layers of the mask network run on conv_walk.cu instead (this kernel remains their
// NHANS_NO_WALK fallback as a plain N = 64 GEMM).
//
// The epilogue is the fusion of blocks.py:104-108 (batch-norm), main.py:166,172 (conditioning adds),
// main.py:184-186 (residual add, ReLU) folded as in SURVEY.md App. A.6.
#include <cstdio>

#include "kernels.h"
#include "ptx.cuh"

namespace nhans {

namespace {

constexpr int kSlabBytes = kSlabRows * 128;       // 17 KB, a multiple of the 1024-byte swizzle atom
constexpr int kCtrlBytes = 8192;
constexpr int kEpiWarps = 8;
constexpr int kEpiWarpBytes = 32 * 64 + 32 * 16;                   // 32 x 16 fp32 transpose buffer + row metadata
constexpr int kEpiBytes = kEpiWarps * kEpiWarpBytes;
constexpr int kMaxGroups = 212;
constexpr int kMaxA = 8, kMaxB = 16;
constexpr int kSmemLimit = 227 * 1024;
constexpr int kWarpA = 8, kWarpB = 9, kWarpMma = 10;

struct __align__(8) Ctrl {
  uint64_t a_full[kMaxA], a_empty[kMaxA];
  uint64_t b_full[kMaxB], b_empty[kMaxB];
  uint64_t tmem_full[2], tmem_empty[2];
  uint32_t tmem_base;
  uint32_t pad;
  KGroupDev groups[kMaxGroups];
};
static_assert(sizeof(Ctrl) <= kCtrlBytes, "control block too large");

// Output row of the tiles one CTA visits (tile0, tile0 + step, ...): ho = (tile / (ksplit n_tiles)) % Ho (kernels.h
// GemmDev), advanced without divisions.
struct TileRow {
  int tpr, d_r, d_ho, Ho, r, ho;
  __device__ __forceinline__ TileRow(int tile0, int step, int tpr_, int Ho_)
      : tpr(tpr_), d_r(step % tpr_), d_ho((step / tpr_) % Ho_), Ho(Ho_), r(tile0 % tpr_), ho((tile0 / tpr_) % Ho_) {}
  __device__ __forceinline__ void next() {
    r += d_r;
    const int carry = r >= tpr ? 1 : 0;
    r -= carry * tpr;
    ho += d_ho + carry;
    if (ho >= Ho) ho -= Ho;
  }
};

// The groups of [g_lo, g_hi) (one K split) a tile runs: [s0, e0) and then [s1, e1), from its row's entry of
// GemmDev::row_groups (empty ranges have e = s)
struct LiveGroups {
  int s0, e0, s1, e1;
  __device__ __forceinline__ LiveGroups(uint32_t w, int g_lo, int g_hi) {
    s0 = max((int)(w & 0xffu), g_lo); e0 = max(s0, min((int)((w >> 8) & 0xffu), g_hi));
    s1 = max((int)((w >> 16) & 0xffu), g_lo); e1 = max(s1, min((int)(w >> 24), g_hi));
  }
};

// MMA issuer (one warp): walks tiles / groups / sub-tiles in the producers' order; one elected lane issues
// tcgen05.mma.  IL sub-tiles are processed together so that consecutive MMAs target different TMEM
// accumulators (back-to-back MMAs into the same accumulator serialise on the accumulate dependency).
// RES: the whole weight matrix is resident in the B ring (towers, small layers); compile-time because every runtime
// test in the single issuing lane's tap loop is paid in throughput (the lane is instruction bound, DESIGN.md §4).
template <int IL, bool CTA2, bool RES>
__device__ __forceinline__ void mma_issuer(Ctrl* ctrl, const GemmDev& p, const GemmCfg& cfg, uint8_t* smem_a, uint8_t* smem_b,
                                           uint32_t tmem_base, int num_tiles, int n_tiles, int b_bytes) {
  const int cta_shift = CTA2 ? 1 : 0;
  const int MT = cfg.mt;
  const int num_groups = p.num_groups;
  // CTA pairs: M = 256 (bit 24.. holds M >> 4), issued by the leader for both CTAs
  const uint32_t idesc = ptx::umma_idesc_f16((uint32_t)p.BN) + (CTA2 ? (8u << 24) : 0u);
  const uint64_t desc_hi = ptx::umma_desc_sw128(0, 0);             // everything but the address field
  const uint32_t a_base = ptx::smem_u32(smem_a) >> 4, b_base = ptx::smem_u32(smem_b) >> 4;
  const uint32_t b_step = (uint32_t)b_bytes >> 4;
  const int gper = (num_groups + p.ksplit - 1) / p.ksplit;      // groups per K split (ksplit = 1: all of them)
  // ONE elected lane runs the whole role - barrier waits, MMAs, commits.  Electing per tap (round 1) cost an
  // elect / branch / warp-sync and a register -> uniform-register shuffle of every descriptor per 4-8 MMAs; in the
  // row-walk kernel the same change was worth 20 %.
  if (ptx::elect_one()) {
    uint32_t aslot = 0, aphase = 0, bslot0 = 0, bphase0 = 0, it = 0;
    uint32_t full_par = 0;                                            // parity of b_full[s] as a group barrier, one bit per slot
    bool b_ready = false;                                             // resident weights have landed
    long long w_tmem = 0, w_a = 0, w_b = 0;
    const bool stats = p.debug_stats != nullptr;                      // wait cycles are only clocked when somebody reads them
    auto wait = [&](uint64_t* bar, uint32_t parity, int tag, long long* acc) {
      if (stats) ptx::mbar_wait_timed(bar, parity, p.err_flag, tag, acc);
      else ptx::mbar_wait(bar, parity, p.err_flag, tag);
    };
    const long long t_start = clock64();
    const int step = gridDim.x >> cta_shift;
    TileRow row(blockIdx.x >> cta_shift, step, p.ksplit * n_tiles, p.Ho);
    for (int tile = blockIdx.x >> cta_shift; tile < num_tiles; tile += step, ++it, row.next()) {
      const uint32_t acc = it & 1, acc_phase = (it >> 1) & 1;
      const int g_lo = (tile % p.ksplit) * gper, g_hi = min(num_groups, g_lo + gper);
      const uint32_t row_w = __ldg(p.row_groups + row.ho);
      wait(&ctrl->tmem_empty[acc], acc_phase ^ 1, 2, &w_tmem);
      ptx::tc_fence_after();
      const LiveGroups lg(row_w, g_lo, g_hi);
      const int g_first = lg.e0 > lg.s0 ? lg.s0 : lg.s1;             // the tile's first MMA overwrites the accumulator
      int gb = lg.s0, ge = lg.e0;
#pragma unroll 1
      for (int pass = 0; pass < 2; ++pass, gb = lg.s1, ge = lg.e1)
      for (int g = gb; g < ge; ++g) {
        const int ntaps = ctrl->groups[g].ntaps;
        // the MT slabs of a group land on the barrier of the group's first slab (MT divides the ring depth, so a
        // group never wraps): one wait per group
        wait(&ctrl->a_full[aslot], aphase, 3, &w_a);
        for (int i0 = 0; i0 < MT; i0 += IL) {
          uint32_t a_lo[IL], d_tm[IL];
#pragma unroll
          for (int ii = 0; ii < IL; ++ii) {
            a_lo[ii] = a_base + (aslot + ii) * (kSlabBytes >> 4);
            d_tm[ii] = tmem_base + acc * 256 + (i0 + ii) * p.BN;
          }
          uint32_t bslot = bslot0, bphase = bphase0;
          if (i0 == 0 && !RES) {
            // every B tile of the group lands on the barrier of the group's first slot: one wait per group
            wait(&ctrl->b_full[bslot0], (full_par >> bslot0) & 1u, 6, &w_b);
            full_par ^= 1u << bslot0;
          }
          for (int t = 0; t < ntaps; ++t) {
            if (RES) {
              bslot = (uint32_t)ctrl->groups[g].bk[t];
              if (!b_ready) wait(&ctrl->b_full[bslot], 0u, 6, &w_b);
            }
            ptx::tc_fence_after();
            const uint32_t sh = (uint32_t)ctrl->groups[g].shift[t] * 8;
            const uint32_t b_lo = b_base + bslot * b_step;
            const uint32_t first = (uint32_t)(g != g_first || t != 0);
            const uint64_t db = desc_hi | b_lo;
#pragma unroll
            for (int k = 0; k < 4; ++k) {                         // +32 B inside the swizzle atom per K = 16
#pragma unroll
              for (int ii = 0; ii < IL; ++ii) {
                if (CTA2) ptx::umma_f16_2sm(d_tm[ii], (desc_hi | (a_lo[ii] + sh)) + 2 * k, db + 2 * k, idesc, k == 0 ? first : 1u);
                else ptx::umma_f16(d_tm[ii], (desc_hi | (a_lo[ii] + sh)) + 2 * k, db + 2 * k, idesc, k == 0 ? first : 1u);
              }
            }
            if (i0 + IL >= MT && !RES) {
              if (CTA2) ptx::umma_commit_2sm(&ctrl->b_empty[bslot]); else ptx::umma_commit(&ctrl->b_empty[bslot]);
            }
            if (!RES && ++bslot == (uint32_t)cfg.nb) { bslot = 0; bphase ^= 1; }
          }
#pragma unroll
          for (int ii = 0; ii < IL; ++ii) {
            if (CTA2) ptx::umma_commit_2sm(&ctrl->a_empty[aslot]); else ptx::umma_commit(&ctrl->a_empty[aslot]);
            if (++aslot == (uint32_t)cfg.na) { aslot = 0; aphase ^= 1; }
          }
          if (i0 + IL >= MT) { bslot0 = bslot; bphase0 = bphase; }
        }
      }
      // resident weights: a tile that ran every group has waited on the barrier of every k-block
      if (lg.e0 - lg.s0 + lg.e1 - lg.s1 == g_hi - g_lo) b_ready = true;
      if (CTA2) ptx::umma_commit_2sm(&ctrl->tmem_full[acc]); else ptx::umma_commit(&ctrl->tmem_full[acc]);
    }
    if (p.debug_stats) {
      atomicAdd(p.debug_stats + 0, (unsigned long long)w_tmem);
      atomicAdd(p.debug_stats + 1, (unsigned long long)w_a);
      atomicAdd(p.debug_stats + 2, (unsigned long long)w_b);
      atomicAdd(p.debug_stats + 4, (unsigned long long)(clock64() - t_start));
    }
  }
  __syncwarp();
}

// Epilogue flavours (compile-time: the epilogue is instruction bound, every runtime flag costs issue slots)
constexpr int kEpiRes = 2;        // + res_scale[c] * x (identity residual)
constexpr int kEpiR1 = 4;         // + r1_vec[c] * raw spectrogram value (1x1 transform with Cin = 1)
constexpr int kEpiTabS = 8;       // time / frequency embedding tables (fp16) resident in shared memory (row flavour)
constexpr int kEpiTabG = 16;      // combined fp32 embedding table read from global memory (transposing flavour)
constexpr int kEpiHead = 32;      // last_dense: fp32 out + centre frame
constexpr int kEpiRow = 64;       // row-per-thread epilogue (below) instead of the transposing one

// One epilogue warp of the BN > 128 layers (a CTA tile is one sub-tile of 128 rows: mt = 1).  ew = 0..7: TMEM lane
// quarter q = ew & 3, and the two warps of a quarter (half = ew >> 2) take alternate 16-column chunks.  Per chunk:
// tcgen05.ld (thread = row) -> XOR-swizzled 32 x 16 fp32 transpose in shared memory -> 4 lanes per row x 4 channels,
// so that global loads / stores are coalesced.  The loads of chunk k + 1 are in flight while chunk k is processed.
template <int EPI, bool CTA2>
__device__ __forceinline__ void epilogue_warp(Ctrl* ctrl, const GemmDev& p, int ew, int lane, uint32_t tmem_base,
                                              int num_tiles, int n_tiles, uint32_t rank) {
  constexpr bool kRes = EPI & kEpiRes, kR1 = EPI & kEpiR1, kTabG = EPI & kEpiTabG, kHead = EPI & kEpiHead;
  const EpiDev& e = p.epi;
  const int q = ew & 3, half = ew >> 2;
  uint8_t* epi_base = reinterpret_cast<uint8_t*>(ctrl) + kCtrlBytes + ew * kEpiWarpBytes;
  uint4* stage = reinterpret_cast<uint4*>(epi_base);                 // [32 rows][4 x 16 B], XOR swizzled
  int4* meta = reinterpret_cast<int4*>(epi_base + 32 * 64);          // [32] {pixel, (ho << 16) | wo, utt, raw bits}
  const int sub = lane >> 2;                // row within a group of 8
  const int jc = lane & 3;                  // 16-byte column slot: channels 4 jc .. 4 jc + 3 of the chunk
  struct LoadSet {
    float4 b[4], t[4];
    uint2 x[4];
  };
  uint32_t it = 0;
  long long w_full = 0;
  const int cta_shift = CTA2 ? 1 : 0;   // CTA pairs: a sub-tile is 256 rows, this CTA owns rows [128 rank, +128)
  const int sub_rows = 128 << cta_shift;
  auto release_acc = [&](uint32_t acc) {      // one arrival per warp on the (leader's) accumulator-free barrier
    ptx::tc_fence_before();
    __syncwarp();
    if (lane == 0) {
      if (CTA2) ptx::mbar_arrive_cluster(&ctrl->tmem_empty[acc], 0);
      else ptx::mbar_arrive(&ctrl->tmem_empty[acc]);
    }
  };
  for (int tile = blockIdx.x >> cta_shift; tile < num_tiles; tile += gridDim.x >> cta_shift, ++it) {
    const uint32_t acc = it & 1, acc_phase = (it >> 1) & 1;
    const int tile_sp = tile / p.ksplit, split = tile - tile_sp * p.ksplit;
    const int n0 = (tile_sp % n_tiles) * p.BN;
    // tile -> (row chunk, image row) with the image row fastest (kernels.h GemmDev)
    const int mtile = tile_sp / n_tiles;
    const int tchunk = mtile / p.Ho, ho = mtile - tchunk * p.Ho;
    const int local0 = tchunk * sub_rows + (int)rank * 128;      // first row of this CTA within the plane
    const int tile_m0 = ho * p.plane_pitch + local0;
    if (local0 >= p.plane_rows) {           // the second CTA of a pair past the plane's last row
      ptx::mbar_wait(&ctrl->tmem_full[acc], acc_phase, p.err_flag, 4);
      release_acc(acc);
      continue;
    }
    // metadata of the row this thread owns (its TMEM lane)
    auto slot_meta = [&]() -> int4 {
      const int r = local0 + q * 32 + lane;
      if (r >= p.plane_rows) return make_int4(-1, 0, 0, 0);
      const int unit = r / p.Wq;
      const int wo = r - unit * p.Wq;
      if (wo >= p.Wo) return make_int4(-1, 0, 0, 0);
      int pix, utt = p.units.utt[unit];
      float rawv = 0.f;
      if (kR1) rawv = epi_raw(e, p.units, unit, ho, wo);
      if (kHead) {
        pix = unit;
        utt = p.units.frame[unit];           // head: the centre frame row replaces the utterance index
      } else if (e.o_mode == 1) {
        pix = (unit * e.o_W + wo) * e.o_H + ho;
      } else {
        pix = (int)epi_grid_pixel(e, unit, ho, wo);
      }
      return make_int4(pix, (ho << 16) | wo, utt, __float_as_int(rawv));
    };
    __syncwarp();
    meta[lane] = slot_meta();
    __syncwarp();
    // per row group g (row 8 g + sub of the warp's 32 rows): element offsets hoisted out of the chunk loop
    bool ok[4];
    float raws[4];
    size_t o_out[4], o_res[4], o_bias[4], o_tf[4];
    const int col0 = n0 + 4 * jc;
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      const int4 mm = meta[g * 8 + sub];
      ok[g] = mm.x >= 0;
      raws[g] = __int_as_float(mm.w);
      const int ho = mm.y >> 16, wo = mm.y & 0xffff;
      o_out[g] = (size_t)mm.x * (kHead ? 201 : e.out_C) + col0;
      o_bias[g] = (size_t)mm.z * (kHead ? 201 : e.bias_stride) + col0;   // head: mm.z = centre frame row of raw
      if (kRes) o_res[g] = (size_t)((long long)tile_m0 + q * 32 + g * 8 + sub) * e.res_C + col0;
      if (kTabG) o_tf[g] = (size_t)(ho * p.Wo + wo) * p.N + col0;
    }
    auto issue_loads = [&](LoadSet& L, int c0) {
      if (kHead || c0 >= p.BN) return;
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        if (!ok[g]) continue;
        L.b[g] = __ldg(reinterpret_cast<const float4*>(e.bias + o_bias[g] + c0));
        if (kTabG) L.t[g] = __ldg(reinterpret_cast<const float4*>(e.tftab + o_tf[g] + c0));
        if (kRes) L.x[g] = __ldg(reinterpret_cast<const uint2*>(e.res + o_res[g] + c0));
      }
    };
    const uint32_t t_addr = tmem_base + ((uint32_t)(q * 32) << 16) + acc * 256;
    auto process = [&](const LoadSet& L, int c0) {
      {
        uint32_t tv[16];
        ptx::tmem_ld16(t_addr + c0, tv);
        ptx::tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 4; ++j)
          stage[lane * 4 + ((j ^ (lane >> 1)) & 3)] = make_uint4(tv[4 * j], tv[4 * j + 1], tv[4 * j + 2], tv[4 * j + 3]);
      }
      __syncwarp();
      float4 rs, r1;
      if (kRes) rs = __ldg(reinterpret_cast<const float4*>(e.res_scale + col0 + c0));
      if (kR1) r1 = __ldg(reinterpret_cast<const float4*>(e.r1_vec + col0 + c0));
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        if (!ok[g]) continue;
        const int r = g * 8 + sub;
        const uint4 u = stage[r * 4 + ((jc ^ (r >> 1)) & 3)];
        float4 f = make_float4(__uint_as_float(u.x), __uint_as_float(u.y), __uint_as_float(u.z), __uint_as_float(u.w));
        if (kHead && p.ksplit > 1) {
          // split-K: raw partial sums of this split, [split][unit][N]; o_out = unit * 201 + col0
          const size_t unit = (o_out[g] - col0) / 201;
          *reinterpret_cast<float4*>(p.split_scratch + ((size_t)split * (p.plane_rows / p.Wq) + unit) * p.N + col0 + c0) = f;
          continue;
        }
        if (kHead) {
          const int col = col0 + c0;
          const float4 b = __ldg(reinterpret_cast<const float4*>(e.bias + col));
          const float4 sc = __ldg(reinterpret_cast<const float4*>(e.res_scale + col));   // inverse weight scale of the column
          const float* raw_row = e.raw + o_bias[g] - col0;
          float* o = e.out_f32 + o_out[g] - col0;
          if (col < 201) o[col] = f.x * sc.x + b.x + raw_row[col];
          if (col + 1 < 201) o[col + 1] = f.y * sc.y + b.y + raw_row[col + 1];
          if (col + 2 < 201) o[col + 2] = f.z * sc.z + b.z + raw_row[col + 2];
          if (col + 3 < 201) o[col + 3] = f.w * sc.w + b.w + raw_row[col + 3];
          continue;
        }
        f.x += L.b[g].x; f.y += L.b[g].y; f.z += L.b[g].z; f.w += L.b[g].w;
        if (kTabG) { f.x += L.t[g].x; f.y += L.t[g].y; f.z += L.t[g].z; f.w += L.t[g].w; }
        if (kRes) {
          const float2 x0 = __half22float2(*reinterpret_cast<const __half2*>(&L.x[g].x));
          const float2 x1 = __half22float2(*reinterpret_cast<const __half2*>(&L.x[g].y));
          f.x = fmaf(rs.x, x0.x, f.x); f.y = fmaf(rs.y, x0.y, f.y);
          f.z = fmaf(rs.z, x1.x, f.z); f.w = fmaf(rs.w, x1.y, f.w);
        }
        if (kR1) {
          f.x = fmaf(r1.x, raws[g], f.x); f.y = fmaf(r1.y, raws[g], f.y);
          f.z = fmaf(r1.z, raws[g], f.z); f.w = fmaf(r1.w, raws[g], f.w);
        }
        if (e.relu) {
          f.x = fmaxf(f.x, 0.f); f.y = fmaxf(f.y, 0.f); f.z = fmaxf(f.z, 0.f); f.w = fmaxf(f.w, 0.f);
        }
        uint2 o;
        o.x = ptx::pack_half2(f.x, f.y);
        o.y = ptx::pack_half2(f.z, f.w);
        *reinterpret_cast<uint2*>(e.out + o_out[g] + c0) = o;
      }
      __syncwarp();                         // staging is overwritten by the next chunk
    };
    // chunks of this warp: the two warps of a quarter alternate 16-column chunks
    LoadSet A, B;
    int c0 = half * 16;
    issue_loads(A, c0);
    ptx::mbar_wait_timed(&ctrl->tmem_full[acc], acc_phase, p.err_flag, 4, &w_full);
    ptx::tc_fence_after();
#pragma unroll 1
    for (; c0 < p.BN; c0 += 64) {
      issue_loads(B, c0 + 32);              // in flight while chunk c0 is processed (no-op past the end)
      process(A, c0);
      if (c0 + 32 < p.BN) {
        issue_loads(A, c0 + 64);
        process(B, c0 + 32);
      }
    }
    release_acc(acc);
  }
  if (p.debug_stats && ew == 0 && lane == 0) atomicAdd(p.debug_stats + 3, (unsigned long long)w_full);
}

// Row-per-thread epilogue.  The transposing epilogue above keeps global accesses coalesced at the price of two
// shared-memory passes per accumulator element; in the 64/128-channel layers those passes compete with the
// tensor core's own operand reads for the shared-memory pipe (ncu: 34 % LSU + 42 % tensor wavefronts, tensor pipe
// 57 % active).  Here a thread keeps the row tcgen05.ld hands it (thread = TMEM lane = GEMM row) and works on 16
// consecutive channels: one 32-byte residual load and one 32-byte store per chunk (256-bit accesses, a full
// sector each), per-channel vectors and the fp16 time / frequency tables from shared memory (frequency rows
// padded by 16 bytes so that the 32 rows of a warp hit different banks), no staging, no metadata exchange.
template <int EPI, bool CTA2>
__device__ __forceinline__ void epilogue_warp_row(Ctrl* ctrl, const GemmDev& p, const GemmCfg& cfg, int ew, int lane,
                                                  uint32_t tmem_base, int num_tiles, int n_tiles, const __half* s_ttab,
                                                  const __half* s_ftab, const float* s_rs, const float* s_r1, uint32_t rank) {
  constexpr bool kRes = EPI & kEpiRes, kR1 = EPI & kEpiR1, kTabS = EPI & kEpiTabS;
  const EpiDev& e = p.epi;
  const int MT = cfg.mt;
  const int q = ew & 3, half = ew >> 2;
  const int f_pitch = p.N + 8;
  struct LoadSet {
    float4 b[4];
    uint4 x[2];
  };
  const int cta_shift = CTA2 ? 1 : 0;
  const int sub_rows = 128 << cta_shift;
  uint32_t it = 0;
  long long w_full = 0;
  auto release_acc = [&](uint32_t acc) {
    ptx::tc_fence_before();
    __syncwarp();
    if (lane == 0) {
      if (CTA2) ptx::mbar_arrive_cluster(&ctrl->tmem_empty[acc], 0);
      else ptx::mbar_arrive(&ctrl->tmem_empty[acc]);
    }
  };
  for (int tile = blockIdx.x >> cta_shift; tile < num_tiles; tile += gridDim.x >> cta_shift, ++it) {
    const uint32_t acc = it & 1, acc_phase = (it >> 1) & 1;
    const int n0 = (tile % n_tiles) * p.BN;
    const int mtile = tile / n_tiles;
    const int tchunk = mtile / p.Ho, ho = mtile - tchunk * p.Ho;      // image row fastest (kernels.h GemmDev)
    const int local0 = tchunk * (MT * sub_rows) + (int)rank * 128;
    const int tile_m0 = ho * p.plane_pitch + local0;
    bool waited = false;
#pragma unroll 1
    for (int i = 0; i < MT; ++i) {
      const int m0 = tile_m0 + i * sub_rows;
      if (local0 + i * sub_rows >= p.plane_rows) break;
      const int m = m0 + q * 32 + lane;
      // the row this thread owns in sub-tile i
      const int r = local0 + i * sub_rows + q * 32 + lane;
      const int unit = r / p.Wq;
      const int wo = r - unit * p.Wq;
      const bool ok = r < p.plane_rows && wo < p.Wo;
      const int utt = ok ? p.units.utt[unit] : 0;
      float rawv = 0.f;
      size_t o_out = 0, o_bias = 0, o_res = 0;
      int o_t = 0, o_f = 0;
      if (ok) {
        if (kR1) rawv = epi_raw(e, p.units, unit, ho, wo);
        o_out = (size_t)epi_pixel(e, unit, ho, wo) * e.out_C + n0;
        o_bias = (size_t)utt * e.bias_stride + n0;
        if (kRes) o_res = (size_t)m * e.res_C + n0;
        if (kTabS) {
          o_t = ho * p.N + n0;
          o_f = wo * f_pitch + n0;
        }
      }
      auto issue_loads = [&](LoadSet& L, int c0) {
        if (c0 >= p.BN || !ok) return;
        const float4* bp = reinterpret_cast<const float4*>(e.bias + o_bias + c0);
        L.b[0] = __ldg(bp); L.b[1] = __ldg(bp + 1); L.b[2] = __ldg(bp + 2); L.b[3] = __ldg(bp + 3);
        if (kRes) ptx::ldg256(e.res + o_res + c0, L.x[0], L.x[1]);
      };
      const uint32_t t_addr = tmem_base + ((uint32_t)(q * 32) << 16) + acc * 256 + i * p.BN;
      auto process = [&](const LoadSet& L, int c0) {
        uint32_t tv[16];
        ptx::tmem_ld16(t_addr + c0, tv);
        ptx::tmem_ld_wait();
        if (!ok) return;
        float f[16];
#pragma unroll
        for (int k = 0; k < 16; ++k) f[k] = __uint_as_float(tv[k]);
#pragma unroll
        for (int k = 0; k < 4; ++k) { f[4 * k] += L.b[k].x; f[4 * k + 1] += L.b[k].y; f[4 * k + 2] += L.b[k].z; f[4 * k + 3] += L.b[k].w; }
        if (kTabS) {
          uint4 tt[2], ff[2];
          tt[0] = *reinterpret_cast<const uint4*>(s_ttab + o_t + c0);
          tt[1] = *reinterpret_cast<const uint4*>(s_ttab + o_t + c0 + 8);
          ff[0] = *reinterpret_cast<const uint4*>(s_ftab + o_f + c0);
          ff[1] = *reinterpret_cast<const uint4*>(s_ftab + o_f + c0 + 8);
          const __half2* th = reinterpret_cast<const __half2*>(tt);
          const __half2* fh = reinterpret_cast<const __half2*>(ff);
#pragma unroll
          for (int k = 0; k < 8; ++k) {
            const float2 s2 = __half22float2(__hadd2(th[k], fh[k]));
            f[2 * k] += s2.x;
            f[2 * k + 1] += s2.y;
          }
        }
        if (kRes) {
          const __half2* xh = reinterpret_cast<const __half2*>(L.x);
          const float4* rs = reinterpret_cast<const float4*>(s_rs + n0 + c0);
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const float4 r = rs[k];
            const float2 x0 = __half22float2(xh[2 * k]), x1 = __half22float2(xh[2 * k + 1]);
            f[4 * k] = fmaf(r.x, x0.x, f[4 * k]); f[4 * k + 1] = fmaf(r.y, x0.y, f[4 * k + 1]);
            f[4 * k + 2] = fmaf(r.z, x1.x, f[4 * k + 2]); f[4 * k + 3] = fmaf(r.w, x1.y, f[4 * k + 3]);
          }
        }
        if (kR1) {
          const float4* r1 = reinterpret_cast<const float4*>(s_r1 + n0 + c0);
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const float4 r = r1[k];
            f[4 * k] = fmaf(r.x, rawv, f[4 * k]); f[4 * k + 1] = fmaf(r.y, rawv, f[4 * k + 1]);
            f[4 * k + 2] = fmaf(r.z, rawv, f[4 * k + 2]); f[4 * k + 3] = fmaf(r.w, rawv, f[4 * k + 3]);
          }
        }
        if (e.relu) {
#pragma unroll
          for (int k = 0; k < 16; ++k) f[k] = fmaxf(f[k], 0.f);
        }
        uint4 o0, o1;
        o0.x = ptx::pack_half2(f[0], f[1]); o0.y = ptx::pack_half2(f[2], f[3]); o0.z = ptx::pack_half2(f[4], f[5]); o0.w = ptx::pack_half2(f[6], f[7]);
        o1.x = ptx::pack_half2(f[8], f[9]); o1.y = ptx::pack_half2(f[10], f[11]); o1.z = ptx::pack_half2(f[12], f[13]); o1.w = ptx::pack_half2(f[14], f[15]);
        ptx::stg256(e.out + o_out + c0, o0, o1);
      };
      LoadSet A, B;
      int c0 = ((half + i) & 1) * 16;
      issue_loads(A, c0);
      if (!waited) {
        ptx::mbar_wait_timed(&ctrl->tmem_full[acc], acc_phase, p.err_flag, 4, &w_full);
        ptx::tc_fence_after();
        waited = true;
      }
#pragma unroll 1
      for (; c0 < p.BN; c0 += 64) {
        issue_loads(B, c0 + 32);
        process(A, c0);
        if (c0 + 32 < p.BN) {
          issue_loads(A, c0 + 64);
          process(B, c0 + 32);
        }
      }
    }
    if (!waited) ptx::mbar_wait(&ctrl->tmem_full[acc], acc_phase, p.err_flag, 4);
    release_acc(acc);
  }
  if (p.debug_stats && ew == 0 && lane == 0) atomicAdd(p.debug_stats + 3, (unsigned long long)w_full);
}

template <int EPI, bool CTA2>
__global__ void __launch_bounds__(kGemmThreads, 1)
gemm_shift_kernel(const __grid_constant__ CUtensorMap mapA0, const __grid_constant__ CUtensorMap mapA1,
                  const __grid_constant__ CUtensorMap mapB, const GemmDev p, const GemmCfg cfg) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = ptx::smem_u32(smem_raw);
  uint8_t* smem = smem_raw + ((1024u - (raw_addr & 1023u)) & 1023u);
  const int cta_shift = CTA2 ? 1 : 0;
  const uint32_t rank = CTA2 ? ptx::cluster_ctarank() : 0u;     // CTA pairs: rank 0 (leader) issues the MMAs
  const int b_bytes = (p.BN >> cta_shift) * 128;                     // a pair splits B: each CTA holds BN / 2 rows
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + cfg.na * kSlabBytes;
  Ctrl* ctrl = reinterpret_cast<Ctrl*>(smem_b + (size_t)cfg.nb * b_bytes);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int MT = cfg.mt;                          // sub-tiles of 128 rows per CTA tile
  const int n_tiles = p.N / p.BN;
  const int tile_rows = (MT * 128) << cta_shift;
  const int m_tiles = p.Ho * ((p.plane_rows + tile_rows - 1) / tile_rows);
  const int num_tiles = m_tiles * n_tiles * p.ksplit;
  const int num_groups = p.num_groups;

  for (int i = threadIdx.x; i < num_groups; i += blockDim.x) ctrl->groups[i] = p.groups[i];
  // row flavour: shared-memory copies of the fp16 time / frequency embedding tables (frequency rows padded by 8
  // halfs), then the per-channel residual scale / rank-1 vectors as fp32, after the control block
  constexpr bool kRow = (EPI & kEpiRow) != 0;
  __half* s_ttab = nullptr;
  __half* s_ftab = nullptr;
  float* s_rs = nullptr;
  float* s_r1 = nullptr;
  if (kRow) {
    uint8_t* tab_base = reinterpret_cast<uint8_t*>(ctrl) + kCtrlBytes;
    float* vec = reinterpret_cast<float*>(tab_base);
    if (EPI & kEpiTabS) {
      const int f_pitch = p.N + 8;
      s_ttab = reinterpret_cast<__half*>(tab_base);
      s_ftab = s_ttab + p.epi.tab_H * p.N;
      vec = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(s_ftab) + (((size_t)p.epi.tab_W * f_pitch * 2 + 15) & ~(size_t)15));
      const int nt = p.epi.tab_H * p.N / 8, c8 = p.N / 8;
      for (int i = threadIdx.x; i < nt; i += blockDim.x) reinterpret_cast<uint4*>(s_ttab)[i] = reinterpret_cast<const uint4*>(p.epi.ttab16)[i];
      for (int i = threadIdx.x; i < p.epi.tab_W * c8; i += blockDim.x) {
        const int w = i / c8, c = i - w * c8;
        *reinterpret_cast<uint4*>(s_ftab + (size_t)w * f_pitch + c * 8) = reinterpret_cast<const uint4*>(p.epi.ftab16)[i];
      }
    }
    s_rs = vec;
    s_r1 = vec + p.N;
    if (EPI & kEpiRes) for (int i = threadIdx.x; i < p.N; i += blockDim.x) s_rs[i] = p.epi.res_scale[i];
    if (EPI & kEpiR1) for (int i = threadIdx.x; i < p.N; i += blockDim.x) s_r1[i] = p.epi.r1_vec[i];
  }
  if (threadIdx.x == 0) {
    for (int s = 0; s < cfg.na; ++s) { ptx::mbar_init(&ctrl->a_full[s], 1); ptx::mbar_init(&ctrl->a_empty[s], 1); }
    for (int s = 0; s < cfg.nb; ++s) { ptx::mbar_init(&ctrl->b_full[s], 1); ptx::mbar_init(&ctrl->b_empty[s], 1); }
    for (int a = 0; a < 2; ++a) {
      ptx::mbar_init(&ctrl->tmem_full[a], 1);
      ptx::mbar_init(&ctrl->tmem_empty[a], kEpiWarps << cta_shift);       // one arrival per epilogue warp (of both CTAs)
    }
    ptx::fence_barrier_init();
    ptx::fence_proxy_async();
  }
  if (warp == kWarpA && lane == 0) {
    ptx::tma_prefetch_desc(&mapA0);
    ptx::tma_prefetch_desc(&mapA1);
    ptx::tma_prefetch_desc(&mapB);
  }
  if (warp == kWarpMma) { if (CTA2) ptx::tmem_alloc_2sm(&ctrl->tmem_base, 512); else ptx::tmem_alloc(&ctrl->tmem_base, 512); }
  ptx::tc_fence_before();
  __syncthreads();
  if (CTA2) ptx::cluster_sync();          // the peer's barriers are initialised before anyone signals them
  ptx::tc_fence_after();
  const uint32_t tmem_base = ctrl->tmem_base;

  // Warp roles: the hardware arbiter favours the highest warp id of a sub-partition, so the single-lane
  // issuers (warps 8-10) out-prioritise the ALU-heavy epilogue warps (0-7) they share a scheduler with.
  if (warp == kWarpA) {
    // ===================== A producer: one slab per (group, sub-tile) =====================
    // (whole warp runs the loop; one elected lane issues the TMA - keeps the control flow warp-uniform)
    uint32_t slot = 0, phase = 0;
    const int gper = (num_groups + p.ksplit - 1) / p.ksplit;
    for (int tile = blockIdx.x >> cta_shift; tile < num_tiles; tile += gridDim.x >> cta_shift) {
      const int mtile = (tile / p.ksplit) / n_tiles;
      const int tchunk = mtile / p.Ho, ho = mtile - tchunk * p.Ho;
      const int m0 = ho * p.plane_pitch + tchunk * tile_rows + (int)rank * 128;
      const int g_lo = (tile % p.ksplit) * gper, g_hi = min(num_groups, g_lo + gper);
      const LiveGroups lg(__ldg(p.row_groups + ho), g_lo, g_hi);      // the issuer's groups, in its order
      int gb = lg.s0, ge = lg.e0;
#pragma unroll 1
      for (int pass = 0; pass < 2; ++pass, gb = lg.s1, ge = lg.e1)
      for (int g = gb; g < ge; ++g) {
        const int row_off = ctrl->groups[g].row_off, col = ctrl->groups[g].col, map = ctrl->groups[g].map;
        uint64_t* gbar = &ctrl->a_full[slot];               // the group's slabs complete on its first slab's barrier
        for (int i = 0; i < MT; ++i) {
          ptx::mbar_wait(&ctrl->a_empty[slot], phase ^ 1, p.err_flag, 1);
          if (ptx::elect_one()) {
            if (CTA2) {
              // both CTAs' slabs are credited to the leader's barrier
              if (rank == 0 && i == 0) ptx::mbar_expect_tx(gbar, 2 * MT * kSlabBytes);
              ptx::tma_load_2d_2sm(smem_a + (size_t)slot * kSlabBytes, map ? &mapA1 : &mapA0, gbar, col,
                                   m0 + i * 256 + row_off);
            } else {
              if (i == 0) ptx::mbar_expect_tx(gbar, MT * kSlabBytes);
              ptx::tma_load_2d(smem_a + (size_t)slot * kSlabBytes, map ? &mapA1 : &mapA0, gbar, col,
                               m0 + i * 128 + row_off);
            }
          }
          __syncwarp();
          if (++slot == (uint32_t)cfg.na) { slot = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == kWarpB) {
    // ===================== B producer =====================
    if (cfg.resident) {
      // the whole packed weight matrix fits: load every k-block once, never release
      for (int t = 0; t < p.num_kb; ++t) {
        if (ptx::elect_one()) {
          ptx::mbar_expect_tx(&ctrl->b_full[t], (uint32_t)b_bytes);
          ptx::tma_load_2d(smem_b + (size_t)t * b_bytes, &mapB, &ctrl->b_full[t], t * 64, 0);
        }
        __syncwarp();
      }
    } else {
      uint32_t slot = 0, phase = 0;
      const int gper = (num_groups + p.ksplit - 1) / p.ksplit;
      const int step = gridDim.x >> cta_shift;
      TileRow row(blockIdx.x >> cta_shift, step, p.ksplit * n_tiles, p.Ho);
      for (int tile = blockIdx.x >> cta_shift; tile < num_tiles; tile += step, row.next()) {
        const int n0 = ((tile / p.ksplit) % n_tiles) * p.BN + (int)rank * (p.BN >> 1) * cta_shift;
        const int g_lo = (tile % p.ksplit) * gper, g_hi = min(num_groups, g_lo + gper);
        const LiveGroups lg(__ldg(p.row_groups + row.ho), g_lo, g_hi);   // the issuer's groups, in its order
        int gb = lg.s0, ge = lg.e0;
#pragma unroll 1
        for (int pass = 0; pass < 2; ++pass, gb = lg.s1, ge = lg.e1)
        for (int g = gb; g < ge; ++g) {
          const int ntaps = ctrl->groups[g].ntaps;
          // all B tiles of a group complete on the barrier of the group's first slot (one wait per group in the issuer)
          uint64_t* gbar = &ctrl->b_full[slot];
          for (int t = 0; t < ntaps; ++t) {
            const int bk = ctrl->groups[g].bk[t];
            ptx::mbar_wait(&ctrl->b_empty[slot], phase ^ 1, p.err_flag, 5);
            if (ptx::elect_one()) {
              if (CTA2) {
                if (rank == 0 && t == 0) ptx::mbar_expect_tx(gbar, 2u * (uint32_t)(ntaps * b_bytes));
                ptx::tma_load_2d_2sm(smem_b + (size_t)slot * b_bytes, &mapB, gbar, bk * 64, n0);
              } else {
                if (t == 0) ptx::mbar_expect_tx(gbar, (uint32_t)(ntaps * b_bytes));
                ptx::tma_load_2d(smem_b + (size_t)slot * b_bytes, &mapB, gbar, bk * 64, n0);
              }
            }
            __syncwarp();
            if (++slot == (uint32_t)cfg.nb) { slot = 0; phase ^= 1; }
          }
        }
      }
    }
  } else if (warp == kWarpMma) {
    // ===================== MMA issuer =====================
    if (rank != 0) {
      // the peer CTA of a pair only lends its shared memory / TMEM; the leader issues for both
    } else if (cfg.resident) {
      if (cfg.il == 2) mma_issuer<2, CTA2, true>(ctrl, p, cfg, smem_a, smem_b, tmem_base, num_tiles, n_tiles, b_bytes);
      else mma_issuer<1, CTA2, true>(ctrl, p, cfg, smem_a, smem_b, tmem_base, num_tiles, n_tiles, b_bytes);
    } else {
      if (cfg.il == 2) mma_issuer<2, CTA2, false>(ctrl, p, cfg, smem_a, smem_b, tmem_base, num_tiles, n_tiles, b_bytes);
      else mma_issuer<1, CTA2, false>(ctrl, p, cfg, smem_a, smem_b, tmem_base, num_tiles, n_tiles, b_bytes);
    }
  } else {
    // ===================== epilogue (warps 0..7) =====================
    if (kRow) epilogue_warp_row<EPI, CTA2>(ctrl, p, cfg, warp, lane, tmem_base, num_tiles, n_tiles, s_ttab, s_ftab, s_rs, s_r1, rank);
    else epilogue_warp<EPI, CTA2>(ctrl, p, warp, lane, tmem_base, num_tiles, n_tiles, rank);
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (CTA2) ptx::cluster_sync();          // nobody exits while the partner may still signal / read it
  if (warp == kWarpMma) {
    __syncwarp();
    ptx::tc_fence_after();
    if (CTA2) ptx::tmem_dealloc_2sm(tmem_base, 512); else ptx::tmem_dealloc(tmem_base, 512);
  }
}

}  // namespace

int gemm_smem_bytes(int BN, int num_kb, int tab_bytes, int cta2, int row, GemmCfg* cfg) {
  const int b_bytes = (cta2 ? BN / 2 : BN) * 128;
  GemmCfg c;
  c.cta2 = cta2;
  c.row = row;
  c.tab_bytes = (tab_bytes + 127) & ~127;       // the row flavour's padded tables + per-channel vectors, else 0
  c.mt = 256 / BN < 1 ? 1 : 256 / BN;
  // A ring: 4 slabs = 4 groups ahead for BN = 256 (one slab per group).  BN <= 128 tiles take two slabs per group and
  // the stride-2 layers consume a group in ~1000 cycles, less than a TMA round trip: 6 slabs (3 groups ahead) cut the
  // issuer's a_full stalls there (B tiles are 8 KB in these layers, the B ring stays >= 9 deep)
  c.na = BN <= 128 ? 6 : 4;
  if (c.na % c.mt != 0) c.na = 4;
  const int epi_bytes = row ? 0 : kEpiBytes;
  const int budget = kSmemLimit - 1024 - kCtrlBytes - epi_bytes - c.tab_bytes - c.na * kSlabBytes;
  c.nb = budget / b_bytes;
  if (c.nb > kMaxB) c.nb = kMaxB;
  c.resident = (num_kb <= c.nb && !cta2) ? 1 : 0;
  c.il = c.mt >= 2 ? 2 : 1;
  if (cfg) *cfg = c;
  return 1024 + c.na * kSlabBytes + c.nb * b_bytes + kCtrlBytes + epi_bytes + c.tab_bytes;
}

namespace {
template <int EPI, bool CTA2>
cudaError_t launch_flavour(cudaStream_t s, int grid, int smem, const CUtensorMap& a0, const CUtensorMap& a1, const CUtensorMap& b,
                           const GemmDev& p, const GemmCfg& cfg) {
  if (CTA2) {
    cudaError_t e2 = cudaFuncSetAttribute(gemm_shift_kernel<EPI, CTA2>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemLimit);
    if (e2 != cudaSuccess) return e2;
    cudaLaunchConfig_t lc{};
    lc.gridDim = dim3(grid);
    lc.blockDim = dim3(kGemmThreads);
    lc.dynamicSmemBytes = smem;
    lc.stream = s;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    lc.attrs = at;
    lc.numAttrs = 1;
    cudaError_t le = cudaLaunchKernelEx(&lc, gemm_shift_kernel<EPI, CTA2>, a0, a1, b, p, cfg);
    if (le != cudaSuccess) {
      int nclusters = -1;
      cudaError_t oe = cudaOccupancyMaxActiveClusters(&nclusters, gemm_shift_kernel<EPI, CTA2>, &lc);
      fprintf(stderr, "nhans: cluster launch failed (%s): grid %d, smem %d, max active clusters %d (%s)\n", cudaGetErrorString(le), grid, smem,
              nclusters, cudaGetErrorString(oe));
    }
    return le;
  }
  cudaError_t e = cudaFuncSetAttribute(gemm_shift_kernel<EPI, CTA2>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemLimit);
  if (e != cudaSuccess) return e;
  gemm_shift_kernel<EPI, CTA2><<<grid, kGemmThreads, smem, s>>>(a0, a1, b, p, cfg);
  return cudaGetLastError();
}
}  // namespace

cudaError_t launch_gemm(cudaStream_t s, int n_sm, const CUtensorMap& mapA0, const CUtensorMap& mapA1,
                        const CUtensorMap& mapB_full, const CUtensorMap& mapB_half, const GemmDev& p) {
  if (p.M <= 0) return cudaSuccess;
  if (p.num_groups > kMaxGroups || !p.row_groups || p.BN % 16 != 0 || p.BN > 256 || p.N % p.BN != 0) return cudaErrorInvalidValue;
  const EpiDev& e = p.epi;
  GemmCfg cfg;
  // row-per-thread epilogue for the 64/128-channel layers, transposing epilogue for BN = 256 and the head
  const int row = (!e.head && p.BN <= 128) ? 1 : 0;
  // the row flavour keeps the fp16 tables (frequency rows padded by 8 halfs) and two per-channel vectors in shared memory
  const bool tabs = e.ttab16 && e.ftab16;
  const int tab_bytes = row ? (tabs ? e.tab_H * p.N * 2 + ((e.tab_W * (p.N + 8) * 2 + 15) & ~15) : 0) + 2 * p.N * 4 : 0;
  // CTA pairs whenever there is enough work for every pair and B splits into two legal boxes
  const int cta2 = ((p.BN % 32) == 0 && !e.head && p.M >= 256 * (n_sm / 2)) ? 1 : 0;
  const int smem = gemm_smem_bytes(p.BN, p.num_kb, tab_bytes, cta2, row, &cfg);
  const CUtensorMap& mapB = cta2 ? mapB_half : mapB_full;
  if (p.N != p.BN) cfg.resident = 0;
  if (cfg.nb < 4 || cfg.na % cfg.mt != 0) return cudaErrorInvalidValue;   // a group has up to 4 taps in flight; its slabs never wrap the A ring
  if (!row && cfg.mt != 1) return cudaErrorInvalidValue;                   // the transposing epilogue handles one sub-tile per tile
  const int tile_rows = (cfg.mt * 128) << cta2;
  if (p.ksplit < 1 || (p.ksplit > 1 && (!e.head || !p.split_scratch || cfg.resident))) return cudaErrorInvalidValue;
  const int tiles = p.Ho * ((p.plane_rows + tile_rows - 1) / tile_rows) * (p.N / p.BN) * p.ksplit;
  int grid = tiles < (n_sm >> cta2) ? tiles : (n_sm >> cta2);
  grid <<= cta2;                              // CTA pairs: two CTAs per tile
  int fl = 0;
  if (e.head) fl = kEpiHead;
  else {
    if (e.res) fl |= kEpiRes;
    if (e.r1_vec) fl |= kEpiR1;
    if (e.tftab) fl |= (row && tabs) ? kEpiTabS : kEpiTabG;
    if (row) fl |= kEpiRow;
  }
#define NHANS_FLAVOUR(F) \
  case F:                \
    return cta2 ? launch_flavour<F, true>(s, grid, smem, mapA0, mapA1, mapB, p, cfg) : launch_flavour<F, false>(s, grid, smem, mapA0, mapA1, mapB, p, cfg);
  switch (fl) {
    NHANS_FLAVOUR(0)                                   // tower layers with 256 / 512 channels, last_conv
    NHANS_FLAVOUR(kEpiTabG)                            // conditioned layers with BN = 256 (tables stay in global memory)
    NHANS_FLAVOUR(kEpiTabG | kEpiRes)
    case kEpiHead:                                     // last_dense (never on CTA pairs)
      return launch_flavour<kEpiHead, false>(s, grid, smem, mapA0, mapA1, mapB, p, cfg);
    NHANS_FLAVOUR(kEpiRow)                             // tower layers with 64 / 128 channels
    NHANS_FLAVOUR(kEpiRow | kEpiR1)                    // tower block-1 conv2
    NHANS_FLAVOUR(kEpiRow | kEpiTabS)                  // conditioned conv1 / conv2 + GEMM transform, BN <= 128
    NHANS_FLAVOUR(kEpiRow | kEpiTabS | kEpiRes)
    NHANS_FLAVOUR(kEpiRow | kEpiTabS | kEpiR1)         // resblock1_1_conv2 without the row-walk kernel
    default: return cudaErrorInvalidValue;
  }
#undef NHANS_FLAVOUR
}

}  // namespace nhans
