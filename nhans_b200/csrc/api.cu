// Engine + C ABI (include/nhans_b200.h): one context per GPU owning a stream, the pre-packed network
// (plan.h) and the batch workspace; runs the STFT -> towers -> conditioned residual stack -> iSTFT path
// of N_HANS___Selective_Noise/apply.py:339-457 for whole batches of utterances with no host round trips
// between the stages.
#include "../../include/nhans_b200.h"

#include <algorithm>
#include <array>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <string>
#include <type_traits>
#include <unordered_map>
#include <unordered_set>
#include <utility>
#include <vector>

#include "kernels.h"
#include "plan.h"

using namespace nhans;

namespace {

thread_local std::string g_create_error;

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// One device allocation, freed by its owner's destructor.
struct DBuf {
  void* p = nullptr;
  size_t cap = 0;
  DBuf() = default;
  DBuf(DBuf&& o) noexcept : p(std::exchange(o.p, nullptr)), cap(std::exchange(o.cap, 0)) {}
  DBuf& operator=(DBuf&& o) noexcept {   // the old allocation goes with `o`
    std::swap(p, o.p);
    std::swap(cap, o.cap);
    return *this;
  }
  ~DBuf() { if (p) cudaFree(p); }
  // replaces the allocation by one of exactly `bytes` (contents not kept)
  cudaError_t alloc(size_t bytes) {
    *this = DBuf();
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e == cudaSuccess) cap = bytes; else p = nullptr;
    return e;
  }
  // at least `bytes`, reallocated with 1/8 of headroom only when too small
  cudaError_t ensure(size_t bytes) { return bytes <= cap ? cudaSuccess : alloc(bytes + bytes / 8 + 256); }
  template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

// Index arrays the library builds on the host (offsets, stream-step descriptors, peaks), sent to the device in one copy.
// add() appends an array at a 16-byte-aligned offset and returns that offset; ptr() is valid only after upload(), which
// may reallocate.  The host bytes stay here until the next use, so the copy never reads from a dead temporary.
struct Staging {
  std::vector<char> host;
  DBuf dev;
  Staging& reset() { host.clear(); return *this; }     // starts a new layout
  template <class T> size_t add(const T* x, size_t n) {
    const size_t off = (host.size() + 15) / 16 * 16;
    host.resize(off + n * sizeof(T));
    if (n) memcpy(host.data() + off, x, n * sizeof(T));
    return off;
  }
  template <class T> size_t add(const std::vector<T>& v) { return add(v.data(), v.size()); }
  cudaError_t upload(cudaStream_t s) {
    cudaError_t e = dev.ensure(host.size());
    return e != cudaSuccess ? e : cudaMemcpyAsync(dev.p, host.data(), host.size(), cudaMemcpyHostToDevice, s);
  }
  template <class T> const T* ptr(size_t off) const { return reinterpret_cast<const T*>(dev.as<char>() + off); }
};

struct GemmLayerDev {
  __half* w = nullptr;
  KGroupDev* groups = nullptr;
  uint32_t* row_groups = nullptr;
  float *bias = nullptr, *tftab = nullptr, *res_scale = nullptr, *r1_vec = nullptr;
  uint16_t *ttab16 = nullptr, *ftab16 = nullptr;
  CUtensorMap mapA0, mapA1, mapB, mapBhalf;
  __half* w_walk = nullptr;         // row-walk layers: weights as [(3 - kh) * 64 + cout][kw * 64 + cin]
  CUtensorMap mapBwalk;
};

struct NetDev {
  NetPlan plan;
  std::vector<__half*> bufs;
  std::vector<GemmLayerDev> layers;
  float *first_w = nullptr, *first_bias = nullptr;
  uint16_t *first_ttab16 = nullptr, *first_ftab16 = nullptr;
  float *Pa = nullptr, *Pb = nullptr, *c = nullptr;
  int *u_frame = nullptr, *u_lo = nullptr, *u_hi = nullptr, *u_utt = nullptr;
  float* convC = nullptr;           // main net: per-frame first-convolution table (kernels.h FrameConvDev)
  float* head_scratch = nullptr;    // main net: split-K partial sums of last_dense [kHeadSplit][capacity][208]
  long long crow_cap = 0;
  std::vector<DBuf> allocs;         // every device allocation above (net_alloc)
  bool ready = false;
};

constexpr int kHeadSplit = 8;       // K splits of last_dense (13312 / 64 = 208 k-blocks -> 26 per split)

struct ProfRec {
  int kind;
  int layer;                        // net * 64 + gemm layer index, or -1
  cudaEvent_t a, b;
  double flops, bytes;
};

// Host <-> device staging of one batch.  There are two sets so that consecutive nhans_enhance_batch calls overlap:
// the H2D copies of batch i + 1 and the D2H copies of batch i - 1 run on their own streams while batch i computes.
struct IoSlot {
  DBuf mix, a, b;
  Staging staging;                  // the batch's Geometry arrays; stage_batch records their device copies below
  const long long *mix_offs = nullptr, *a_offs = nullptr, *b_offs = nullptr, *frame_offs = nullptr, *out_offs = nullptr,
                  *ctx_frame_offs = nullptr;
  DBuf out_i16, out_f32;
  cudaEvent_t uploaded = nullptr;   // h2d stream: inputs of the batch staged in this set have landed
  cudaEvent_t consumed = nullptr;   // compute stream: every kernel reading / writing this set has finished
  cudaEvent_t drained = nullptr;    // d2h stream: outputs of this set have reached the host
  bool d2h_pending = false;
};

// Layout of a batch of U utterances (batch_geometry).  Sample offsets are relative to the first sample of each array;
// a_offs / b_offs are empty when the batch has no such context.
struct Geometry {
  int U = 0;
  std::vector<long long> mix_offs;  // [u < U]: first sample of utterance u's kept frames; [U]: samples in the array
  std::vector<long long> a_offs, b_offs;
  std::vector<long long> frame_offs, out_offs;   // kept mixture frames and output samples of each utterance
  std::vector<long long> ctx_frame_offs;         // u * 200: the context frames the towers read
  int max_frames = 0;
  long long total_frames = 0, total_out = 0;
};

// Conditioning of U context pairs (run_conditioning): peaks of int16 clips, the first 200 STFT frames of each clip,
// their embeddings and the conditioning table [U][n_cols].
struct CondBufs {
  DBuf peak_a, peak_b, ctxlm_a, ctxlm_b, emb_a, emb_b, cond;
};

struct Batch {
  Geometry geo;
  bool has_a = false;
  bool staged = false, done = false;
  IoSlot io[2];
  int cur = 0;                      // set the staged / running batch uses
  DBuf peak_mix;
  CondBufs cb;
  DBuf logmag, phase, den, mixproc, removed, comp, sums, snr;
};

// Host side of one open stream (nhans_stream_open).  Its device state is slot `slot` of Streams::pool
// (kernels.h StreamStepDev): the conditioning row, the last <= 34 frames (log-magnitude and phasors) its next windows
// read, and its last two denoised frames.
struct StreamRec {
  int slot = -1, peak = 0;
  bool final = false;               // the final step has run: no further chunks
  long long n = 0;                  // samples received
  std::vector<int16_t> tail;        // samples from 160 * frames_of(n) on, where the next frame starts
  double e_den = 0, e_rem = 0;      // sum den^2, sum removed^2 of the samples emitted by nhans_stream_step_post
};

// Every open stream of a context, with device buffers of their own (the batch path's results stay untouched).
struct Streams {
  std::unordered_map<int, StreamRec> rec;
  int next_id = 0;
  DBuf pool;                        // slots of slot_stride floats
  int n_slots = 0;
  long long slot_stride = 0;
  std::vector<int> free_slots;
  DBuf ctx_a, ctx_b;                // nhans_stream_open
  CondBufs cb;
  DBuf pcm, new_lm, new_ph, seg_lm, seg_ph, den_win, den_seg, cond, out_i16, out_f32;   // nhans_stream_step
  DBuf mixed, removed, comp, sums;                                                     // nhans_stream_step_post
};

}  // namespace

struct nhans_ctx {
  int device = 0, variant = 0;
  int win_cap = 2048, row_cap = 32;
  int n_sm = 148;
  cudaStream_t stream = nullptr;    // compute
  cudaStream_t h2d_stream = nullptr, d2h_stream = nullptr;
  std::string err;
  std::string json;
  EncodeTiledFn encode = nullptr;
  NetDev main_net, tower;
  int* err_flag_host = nullptr;     // mapped pinned: written by a kernel that gave up waiting
  int* err_flag_dev = nullptr;
  DBuf silent_emb;
  bool silent_ready = false;
  Batch batch;
  Streams streams;
  DBuf tmp[8];
  Staging staging;                  // index arrays of the calls that finish before they return (all but the batch path)
  cudaEvent_t events[16] = {};
  bool profile = false;
  std::vector<ProfRec> prof;
  std::vector<cudaEvent_t> ev_pool;
  double prof_acc[5][4] = {};
  unsigned long long* debug_stats = nullptr;   // [128][8] per-layer wait-cycle counters (NHANS_DEBUG_STATS=1)
  // NHANS_DEBUG_TIMELINE=1: timing events on the three streams for every batch (nhans_debug_timeline)
  bool timeline = false;
  cudaEvent_t tl_origin = nullptr;
  std::vector<std::array<cudaEvent_t, 6>> tl;     // per batch: h2d begin / end, compute begin / end, d2h begin / end
  bool use_walk = true;             // row-walk kernel for the 64-channel stage (NHANS_NO_WALK=1: plain N = 64 GEMM)
  bool use_gen = true;              // resblock1_1_conv2 builds its A operand from the per-frame table (NHANS_NO_GEN=1: window_expand)
  double layer_acc[128][4] = {};
  double launches = 0;              // every kernel launched by this context (counted even when not profiling)
  // Also runs on a context nhans_create gave up on, whose later handles are still null.  The device buffers go with
  // their DBufs.
  ~nhans_ctx() {
    for (IoSlot& io : batch.io)
      for (cudaEvent_t ev : {io.uploaded, io.consumed, io.drained}) if (ev) cudaEventDestroy(ev);
    for (cudaEvent_t ev : events) if (ev) cudaEventDestroy(ev);
    for (auto& r : prof) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
    for (cudaEvent_t ev : ev_pool) cudaEventDestroy(ev);
    for (auto& t : tl) for (cudaEvent_t ev : t) if (ev) cudaEventDestroy(ev);
    if (tl_origin) cudaEventDestroy(tl_origin);
    if (err_flag_host) cudaFreeHost(err_flag_host);
    if (debug_stats) cudaFree(debug_stats);
    for (cudaStream_t s : {stream, h2d_stream, d2h_stream}) if (s) cudaStreamDestroy(s);
  }
};

namespace {

int fail(nhans_ctx* c, int code, const std::string& msg) {
  if (c) c->err = msg;
  return code;
}

#define CK(call)                                                                                         \
  do {                                                                                                   \
    cudaError_t e__ = (call);                                                                            \
    if (e__ != cudaSuccess)                                                                              \
      return fail(ctx, NHANS_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__) + " (" + __FILE__ + ":" + \
                                           std::to_string(__LINE__) + ")");                              \
  } while (0)

// Every launcher call goes through here: its result is checked and the launch counted in ctx->launches
// (nhans_profile_get kind 5).  `what` names the launch in the error and is built only on failure.
#define LAUNCH_AS(call, what)                                                                            \
  do {                                                                                                   \
    cudaError_t e__ = (call);                                                                            \
    if (e__ != cudaSuccess) return fail(ctx, NHANS_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e__)); \
    ctx->launches += 1;                                                                                  \
  } while (0)
#define LAUNCH(call) LAUNCH_AS(call, std::string(#call) + " (" + __FILE__ + ":" + std::to_string(__LINE__) + ")")

// n elements of device memory owned by `net`, zeroed on the compute stream when `zero`.
template <class T>
int net_alloc(nhans_ctx* ctx, NetDev& net, size_t n, T** out, bool zero = false) {
  net.allocs.emplace_back();
  DBuf& d = net.allocs.back();
  CK(d.alloc(n * sizeof(T)));
  if (zero) CK(cudaMemsetAsync(d.p, 0, n * sizeof(T), ctx->stream));
  *out = d.as<T>();
  return 0;
}

template <class T>
int upload(nhans_ctx* ctx, NetDev& net, const std::vector<T>& h, T** out) {
  *out = nullptr;
  if (h.empty()) return 0;
  if (int rc = net_alloc(ctx, net, h.size(), out)) return rc;
  CK(cudaMemcpyAsync(*out, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
  return 0;
}

int make_map(nhans_ctx* ctx, CUtensorMap* map, const void* base, long long cols, long long rows, int box_rows) {
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)cols * 2};
  cuuint32_t box[2] = {64u, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1u, 1u};
  CUresult r = ctx->encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return fail(ctx, NHANS_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult " + std::to_string((int)r) + " (cols " +
                                         std::to_string(cols) + ", rows " + std::to_string(rows) + ")");
  return 0;
}

// Allocates the activation grids (zeroed once: padding positions are never written afterwards), uploads
// packed weights and epilogue tables, encodes the TMA descriptors.
int realise_net(nhans_ctx* ctx, NetDev& net) {
  const NetPlan& P = net.plan;
  int rc;
  net.bufs.assign(P.bufs.size(), nullptr);
  for (size_t i = 0; i < P.bufs.size(); ++i)
    if ((rc = net_alloc(ctx, net, (size_t)P.bufs[i].pixels * P.bufs[i].C, &net.bufs[i], true))) return rc;
  if (P.cond.n_cols > 0) {
    // main net: its first convolution runs once per frame (kernels.h FrameConvDev), which needs this shape
    const DirectLayer& D = P.first;
    if (D.kh != 4 || D.kw != 4 || D.sh != 1 || D.sw != 1 || D.pt != 1 || D.pl != 1 || D.Hin != kWinFrames || D.Ho != kWinFrames ||
        D.raw_oh != -(kWinFrames / 2) || D.N != 64)
      return fail(ctx, NHANS_ERR_STATE, "first convolution of the mask network with an unexpected shape");
    // per-frame table: a pass's windows plus kWinReach virtual frames per utterance it touches.  run_masknet sizes every pass
    // to fit, so utterances that average fewer than 17 frames run in smaller passes.
    net.crow_cap = 3LL * P.capacity + 64;
    if ((rc = net_alloc(ctx, net, (size_t)4 * net.crow_cap * kBins * 64, &net.convC))) return rc;
  }
  if (P.cond.n_cols > 0 && !P.gemm.empty() && P.gemm.back().epi.head && !getenv("NHANS_NO_SPLITK"))
    if ((rc = net_alloc(ctx, net, (size_t)kHeadSplit * P.capacity * P.gemm.back().N, &net.head_scratch))) return rc;
  if ((rc = upload(ctx, net, P.first.w, &net.first_w))) return rc;
  if ((rc = upload(ctx, net, P.first.epi.bias, &net.first_bias))) return rc;
  if ((rc = upload(ctx, net, P.first.epi.ttab16, &net.first_ttab16))) return rc;
  if ((rc = upload(ctx, net, P.first.epi.ftab16, &net.first_ftab16))) return rc;
  if ((rc = upload(ctx, net, P.cond.Pa, &net.Pa))) return rc;
  if ((rc = upload(ctx, net, P.cond.Pb, &net.Pb))) return rc;
  if ((rc = upload(ctx, net, P.cond.c, &net.c))) return rc;
  net.layers.resize(P.gemm.size());
  for (size_t i = 0; i < P.gemm.size(); ++i) {
    const GemmLayer& L = P.gemm[i];
    GemmLayerDev& D = net.layers[i];
    uint16_t* dw = nullptr;
    if ((rc = upload(ctx, net, L.w, &dw))) return rc;
    D.w = reinterpret_cast<__half*>(dw);
    std::vector<KGroupDev> groups(L.groups.size());
    for (size_t j = 0; j < groups.size(); ++j) {
      const KGroup& g = L.groups[j];
      KGroupDev d;
      d.row_off = g.row_off; d.map = g.map; d.col = g.col; d.ntaps = g.ntaps; d.pad_ = 0;
      for (int t = 0; t < 4; ++t) { d.shift[t] = g.shift[t]; d.bk[t] = g.bk[t]; }
      groups[j] = d;
    }
    if ((rc = upload(ctx, net, groups, &D.groups))) return rc;
    if ((rc = upload(ctx, net, L.row_groups, &D.row_groups))) return rc;
    if (L.epi.head && (int)L.groups.size() % kHeadSplit == 0 && !every_split_live(L, kHeadSplit))
      return fail(ctx, NHANS_ERR_STATE, "layer " + L.name + ": a K split runs no group for some output row");
    if ((rc = upload(ctx, net, L.epi.bias, &D.bias))) return rc;
    if ((rc = upload(ctx, net, L.epi.tftab, &D.tftab))) return rc;
    if ((rc = upload(ctx, net, L.epi.ttab16, &D.ttab16))) return rc;
    if ((rc = upload(ctx, net, L.epi.ftab16, &D.ftab16))) return rc;
    if ((rc = upload(ctx, net, L.epi.res_scale, &D.res_scale))) return rc;
    if ((rc = upload(ctx, net, L.epi.r1_vec, &D.r1_vec))) return rc;
    for (int a = 0; a < 2; ++a) {
      int buf = L.a_buf[a] >= 0 ? L.a_buf[a] : L.a_buf[0];
      int rowlen = L.a_buf[a] >= 0 ? L.a_rowlen[a] : L.a_rowlen[0];
      const Grid& g = P.bufs[buf];
      long long elems = (long long)g.pixels * g.C;
      if (elems % rowlen) return fail(ctx, NHANS_ERR_STATE, "buffer size not a multiple of the TMA row length");
      if ((rc = make_map(ctx, a == 0 ? &D.mapA0 : &D.mapA1, net.bufs[buf], rowlen, elems / rowlen, kSlabRows))) return rc;
    }
    if ((rc = make_map(ctx, &D.mapB, D.w, L.K, L.N, L.BN))) return rc;
    if ((rc = make_map(ctx, &D.mapBhalf, D.w, L.K, L.N, L.BN % 32 == 0 ? L.BN / 2 : L.BN))) return rc;   // CTA pairs load half of B each
    if (L.walk) {
      if (L.c_kh != 4 || L.c_kw != 4 || L.N != 64 || L.K != 16 * 64) return fail(ctx, NHANS_ERR_STATE, "row-walk layer with an unexpected shape");
      std::vector<uint16_t> ww((size_t)256 * 256);
      for (int kh = 0; kh < 4; ++kh)
        for (int kw = 0; kw < 4; ++kw)
          for (int co = 0; co < 64; ++co)
            for (int ci = 0; ci < 64; ++ci)
              ww[(size_t)((3 - kh) * 64 + co) * 256 + kw * 64 + ci] = L.w[(size_t)co * L.K + (kh * 4 + kw) * 64 + ci];
      if ((rc = upload(ctx, net, ww, &dw))) return rc;
      CK(cudaStreamSynchronize(ctx->stream));          // `ww` is a temporary
      D.w_walk = reinterpret_cast<__half*>(dw);
      if ((rc = make_map(ctx, &D.mapBwalk, D.w_walk, 256, 256, 256))) return rc;
    }
  }
  for (int** p : {&net.u_frame, &net.u_lo, &net.u_hi, &net.u_utt})
    if ((rc = net_alloc(ctx, net, P.capacity, p))) return rc;
  CK(cudaStreamSynchronize(ctx->stream));
  net.ready = true;
  return 0;
}

// ---- profiling -----------------------------------------------------------------------------------
cudaEvent_t get_event(nhans_ctx* ctx) {
  if (!ctx->ev_pool.empty()) {
    cudaEvent_t e = ctx->ev_pool.back();
    ctx->ev_pool.pop_back();
    return e;
  }
  cudaEvent_t e = nullptr;
  cudaEventCreate(&e);
  return e;
}

struct ProfScope {
  nhans_ctx* ctx;
  bool on;
  ProfRec r;
  ProfScope(nhans_ctx* c, int kind, double flops, double bytes, int layer = -1) : ctx(c), on(c->profile) {
    if (!on) return;
    r.kind = kind; r.flops = flops; r.bytes = bytes; r.layer = layer;
    r.a = get_event(c); r.b = get_event(c);
    cudaEventRecord(r.a, c->stream);
  }
  ~ProfScope() {
    if (!on) return;
    cudaEventRecord(r.b, ctx->stream);
    ctx->prof.push_back(r);
  }
};

void prof_collect(nhans_ctx* ctx) {
  if (ctx->prof.empty()) return;
  cudaStreamSynchronize(ctx->stream);
  for (auto& r : ctx->prof) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, r.a, r.b) == cudaSuccess) {
      double* a = ctx->prof_acc[r.kind];
      a[0] += 1; a[1] += ms; a[2] += r.flops; a[3] += r.bytes;
      if (r.layer >= 0 && r.layer < 128) {
        double* l = ctx->layer_acc[r.layer];
        l[0] += 1; l[1] += ms; l[2] += r.flops; l[3] += r.bytes;
      }
    }
    ctx->ev_pool.push_back(r.a);
    ctx->ev_pool.push_back(r.b);
  }
  ctx->prof.clear();
}

// ---- network execution ---------------------------------------------------------------------------
void fill_out(EpiDev& e, const NetDev& net, const Grid& g) {
  e.out = g.buf >= 0 ? net.bufs[g.buf] : nullptr;
  e.out_C = g.C;
  e.o_mode = g.mode; e.o_sh = g.sh; e.o_sw = g.sw; e.o_oy = g.oy; e.o_ox = g.ox;
  e.o_H = g.H; e.o_W = g.W;
  e.o_plane = g.plane_stride; e.o_rstride = g.rstride; e.o_ustride = g.ustride;
}

EpiDev make_epi(const NetDev& net, const Epilogue& E, const Grid& out, const float* bias_const, const float* tftab,
                const float* res_scale, const float* r1_vec, const float* raw, const float* cond_table,
                float* out_f32) {
  EpiDev e;
  memset(&e, 0, sizeof e);
  if (E.cond_off >= 0) {
    e.bias = cond_table + E.cond_off;
    e.bias_stride = net.plan.cond.n_cols;
  } else {
    e.bias = bias_const;
    e.bias_stride = 0;
  }
  e.tftab = tftab;
  if (E.res_buf >= 0) {
    e.res = net.bufs[E.res_buf];
    e.res_C = net.plan.bufs[E.res_buf].C;
    e.res_scale = res_scale;
  }
  if (E.head) e.res_scale = res_scale;      // head: inverse of the per-column weight scale
  e.r1_vec = r1_vec; e.r1_sh = E.r1_sh; e.r1_sw = E.r1_sw; e.raw_oh = E.raw_oh;
  e.raw = raw;
  e.relu = E.relu; e.head = E.head;
  fill_out(e, net, out);
  e.out_f32 = out_f32;
  return e;
}

struct PassInfo {                   // which utterances / per-frame table rows a pass of the mask network touches
  const long long* d_frame_offs;
  int u_first, u_last;
  long long crow0;                  // first table row = frame of the first window + kWinReach * u_first
  int rows;                         // table rows of the pass (<= crow_cap)
};

// Runs `units` windows / context rows whose unit tables are already filled.
int run_net(nhans_ctx* ctx, NetDev& net, int units, const float* raw, const float* cond_table, float* out_f32,
            const PassInfo* pass = nullptr) {
  const NetPlan& P = net.plan;
  UnitTable ut{net.u_frame, net.u_lo, net.u_hi, net.u_utt};
  bool gen_first = false;
  {
    const DirectLayer& D = P.first;
    DirectDev d;
    memset(&d, 0, sizeof d);
    d.units = units;
    d.kh = D.kh; d.kw = D.kw; d.sh = D.sh; d.sw = D.sw; d.pt = D.pt; d.pl = D.pl;
    d.Hin = D.Hin; d.Win = D.Win; d.raw_oh = D.raw_oh; d.Ho = D.Ho; d.Wo = D.Wo; d.N = D.N;
    d.w = net.first_w;
    d.units_tab = ut;
    d.epi = make_epi(net, D.epi, D.out, net.first_bias, nullptr, nullptr, nullptr, raw, cond_table, nullptr);
    d.epi.ttab16 = reinterpret_cast<const __half*>(net.first_ttab16);
    d.epi.ftab16 = reinterpret_cast<const __half*>(net.first_ftab16);
    d.epi.tab_H = D.Ho; d.epi.tab_W = D.Wo;
    ProfScope ps(ctx, 3, 2.0 * D.macs_per_unit * units, 0);
    if (pass) {
      FrameConvDev f;
      memset(&f, 0, sizeof f);
      f.raw = raw; f.frame_offs = pass->d_frame_offs;
      f.u_first = pass->u_first; f.u_last = pass->u_last;
      f.crow0 = pass->crow0;
      f.rows = pass->rows;
      f.crow_cap = net.crow_cap;
      f.w = net.first_w;
      f.bias = d.epi.bias; f.bias_stride = d.epi.bias_stride; f.ftab16 = d.epi.ftab16;
      f.C = net.convC;
      // (expanding the pass in slices so that a slice's table stays L2-resident was measured: no gain)
      LAUNCH(launch_frame_conv(ctx->stream, f));
      // the row-walk kernel of the next layer builds its A operand from the table (conv_walk.cu kWalkGen); otherwise
      // the table is expanded into the (window, row) activation tensor here
      gen_first = ctx->use_walk && ctx->use_gen && !P.gemm.empty() && P.gemm[0].walk && net.layers[0].w_walk &&
                  P.gemm[0].a_buf[0] == D.out.buf && D.epi.relu && d.epi.ttab16;
      if (!gen_first) LAUNCH(launch_window_expand(ctx->stream, d, net.convC, pass->crow0, net.crow_cap, 0, units));
    } else {
      LAUNCH(launch_direct_conv(ctx->stream, d));
    }
  }
  for (size_t i = 0; i < P.gemm.size(); ++i) {
    const GemmLayer& L = P.gemm[i];
    const GemmLayerDev& D = net.layers[i];
    GemmDev g;
    memset(&g, 0, sizeof g);
    long long M = (long long)units * L.Ho * L.Wq;
    if ((long long)P.capacity * L.Ho * L.Wq > 0x7fffffffLL) return fail(ctx, NHANS_ERR_ARG, "too many rows in one pass");
    g.M = (int)M; g.plane_pitch = P.capacity * L.Wq; g.plane_rows = units * L.Wq; g.N = L.N; g.BN = L.BN; g.num_kb = (int)L.kb.size(); g.num_groups = (int)L.groups.size(); g.groups = D.groups; g.row_groups = D.row_groups;
    g.Hq = L.Hq; g.Wq = L.Wq; g.Ho = L.Ho; g.Wo = L.Wo;
    g.units = ut;
    g.epi = make_epi(net, L.epi, L.out, D.bias, D.tftab, D.res_scale, D.r1_vec, raw, cond_table, out_f32);
    g.epi.ttab16 = reinterpret_cast<const __half*>(D.ttab16);
    g.epi.ftab16 = reinterpret_cast<const __half*>(D.ftab16);
    g.epi.tab_H = L.Ho;
    g.epi.tab_W = L.Wo;
    g.err_flag = ctx->err_flag_dev;
    g.ksplit = 1;
    // last_dense: 16 row tiles per 2048-window pass but K = 13312 - split K over the idle SMs (deterministic two-stage sum)
    // (whatever the pass size: the summation order - and with it every output bit - must not depend on how many windows
    // share the pass)
    const bool split_head = L.epi.head && net.head_scratch && (int)L.groups.size() % kHeadSplit == 0;
    if (split_head) { g.ksplit = kHeadSplit; g.split_scratch = net.head_scratch; }
    g.debug_stats = ctx->debug_stats ? ctx->debug_stats + 8 * ((&net == &ctx->tower ? 64 : 0) + (int)i) : nullptr;
    ProfScope ps(ctx, 0, 2.0 * L.macs_per_unit * units, 0, (&net == &ctx->tower ? 64 : 0) + (int)i);
    if (L.walk && D.w_walk && ctx->use_walk) {
      WalkDev wd;
      memset(&wd, 0, sizeof wd);
      wd.plane_pitch = g.plane_pitch; wd.plane_rows = g.plane_rows;
      wd.H = L.Ho; wd.Wq = L.Wq; wd.Wo = L.Wo; wd.pt = L.c_pt; wd.pl = L.c_pl;
      wd.units = ut; wd.epi = g.epi; wd.err_flag = g.err_flag; wd.debug_stats = g.debug_stats;
      if (i == 0 && gen_first) {
        wd.gen_C = net.convC; wd.gen_crow0 = pass->crow0; wd.gen_crow_cap = net.crow_cap;
        wd.gen_ttab16 = reinterpret_cast<const __half*>(net.first_ttab16);
      }
      LAUNCH_AS(launch_walk(ctx->stream, ctx->n_sm, D.mapA0, D.mapBwalk, wd), "launch of row-walk layer " + L.name);
      continue;
    }
    LAUNCH_AS(launch_gemm(ctx->stream, ctx->n_sm, D.mapA0, D.mapA1, D.mapB, D.mapBhalf, g),
              "launch of layer " + L.name + " (M " + std::to_string(g.M) + ", BN " + std::to_string(g.BN) + ")");
    if (split_head)
      LAUNCH(launch_head_reduce(ctx->stream, net.head_scratch, kHeadSplit, units, L.N, D.res_scale, D.bias, raw, net.u_frame, out_f32));
  }
  return 0;
}

// Embedding tower over R context rows of ctx_logmag (device, [R][200][201]) -> emb (device, [R][512]).
int run_tower(nhans_ctx* ctx, const float* ctx_logmag, int R, float* emb) {
  NetDev& net = ctx->tower;
  const int cap = net.plan.capacity;
  for (int r0 = 0; r0 < R; r0 += cap) {
    const int n = std::min(cap, R - r0);
    LAUNCH(launch_units_rows(ctx->stream, r0, n, kCtxFrames, net.u_frame, net.u_lo, net.u_hi, net.u_utt));
    int rc = run_net(ctx, net, n, ctx_logmag, nullptr, nullptr);
    if (rc) return rc;
    ProfScope ps(ctx, 4, 0, 0);
    LAUNCH(launch_mean_pool(ctx->stream, net.bufs[net.plan.pool_buf], n, net.plan.pool_pixels, 512, emb + (size_t)r0 * 512));
  }
  return 0;
}

// Mask network over windows -> denoised rows den[window].  Segment s stores frames [frame_offs[s], frame_offs[s + 1]) of
// `logmag` (rows outside read as zero padding) and owns windows [win_offs[s], win_offs[s + 1]), centred on stored frames
// frame_offs[s] + left[s] + ...  A whole utterance has one window per frame: win_offs = frame_offs and left = null.
int run_masknet(nhans_ctx* ctx, const float* logmag, const long long* d_frame_offs, const long long* h_frame_offs,
                const long long* d_win_offs, const long long* h_win_offs, const int* d_left, const int* h_left, int U,
                const float* cond_table, float* den) {
  NetDev& net = ctx->main_net;
  const int cap = net.plan.capacity;
  const long long total_windows = h_win_offs[U];
  if (h_frame_offs[U] > 0x7fffffffLL) return fail(ctx, NHANS_ERR_ARG, "too many frames in one batch");
  // segment of a window: largest s with win_offs[s] <= window
  auto seg_of = [&](long long w) { return (int)(std::upper_bound(h_win_offs, h_win_offs + U + 1, w) - h_win_offs) - 1; };
  // per-frame table row of window row 0 of window w (kernels.h FrameConvDev: stored frame + kWinReach per earlier segment)
  auto crow_of = [&](long long w) {
    const int s = seg_of(w);
    return h_frame_offs[s] + (h_left ? h_left[s] : 0) + (w - h_win_offs[s]) + (long long)kWinReach * s;
  };
  for (long long w0 = 0, n = 0; w0 < total_windows; w0 += n) {
    PassInfo pi;
    pi.d_frame_offs = d_frame_offs;
    pi.u_first = seg_of(w0);
    pi.crow0 = crow_of(w0);
    // the largest pass whose per-frame table rows fit; one window always does.  For whole utterances these are its
    // windows + kWinReach per utterance.
    auto rows = [&](long long m) { return crow_of(w0 + m - 1) + 35 - pi.crow0; };
    long long lo = 1, hi = std::min<long long>(cap, total_windows - w0);
    while (lo < hi) {
      const long long mid = (lo + hi + 1) / 2;
      if (rows(mid) <= net.crow_cap) lo = mid; else hi = mid - 1;
    }
    n = lo;
    pi.u_last = seg_of(w0 + n - 1);
    pi.rows = (int)rows(n);
    LAUNCH(launch_units_main(ctx->stream, d_frame_offs, d_win_offs, d_left, U, (int)w0, (int)n, net.u_frame, net.u_lo,
                             net.u_hi, net.u_utt));
    int rc = run_net(ctx, net, (int)n, logmag, cond_table, den + (size_t)w0 * kBins, &pi);
    if (rc) return rc;
  }
  return 0;
}

int ensure_silent(nhans_ctx* ctx) {
  if (ctx->silent_ready) return 0;
  // Silent.wav (SN/apply.py:479-480) is all zeros: log(0 + 1e-5) in every bin of all 200 frames.
  std::vector<float> row((size_t)kCtxFrames * kBins, logf(1e-5f));
  CK(ctx->tmp[7].ensure(row.size() * 4));
  CK(cudaMemcpyAsync(ctx->tmp[7].p, row.data(), row.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
  CK(ctx->silent_emb.ensure(512 * 4));
  int rc = run_tower(ctx, ctx->tmp[7].as<float>(), 1, ctx->silent_emb.as<float>());
  if (rc) return rc;
  CK(cudaStreamSynchronize(ctx->stream));
  ctx->silent_ready = true;
  return 0;
}

// timeline: record timing event `which` of the newest batch on `stream`
void tl_mark(nhans_ctx* ctx, int which, cudaStream_t stream) {
  if (!ctx->timeline) return;
  if (!ctx->tl_origin) {
    cudaEventCreate(&ctx->tl_origin);
    cudaEventRecord(ctx->tl_origin, stream);
  }
  if (which == 0) {
    std::array<cudaEvent_t, 6> ev{};
    for (auto& e : ev) cudaEventCreate(&e);
    ctx->tl.push_back(ev);
  }
  if (ctx->tl.empty()) return;
  cudaEventRecord(ctx->tl.back()[which], stream);
}

int check_kernel_flag(nhans_ctx* ctx) {
  if (ctx->err_flag_host && *ctx->err_flag_host) {
    // reported once: the flag is cleared so that a later call (after nhans_load_weights, or on a context whose
    // launch merely failed) is judged on its own; a trapped kernel leaves the CUDA context unusable anyway
    const int tag = *ctx->err_flag_host;
    *ctx->err_flag_host = 0;
    return fail(ctx, NHANS_ERR_KERNEL, "tensor-core pipeline timed out waiting on barrier class " + std::to_string(tag));
  }
  return 0;
}

// Result of a call after waiting on its work (e): a kernel that gave up waiting explains the CUDA error it leaves.
int finish(nhans_ctx* ctx, cudaError_t e) {
  if (int rc = check_kernel_flag(ctx)) return rc;
  CK(e);
  return NHANS_OK;
}

int frames_of(long long n) { return n >= 400 ? (int)(1 + (n - 400) / 160) : 0; }

// samples the inverse STFT returns for T frames
long long out_len(long long T) { return T > 0 ? (T - 1) * 160 + 400 : 0; }

constexpr int kWholeClips = -1;     // batch_geometry: keep every frame, and allow mixtures shorter than one frame

// Lays out a batch from the caller's sample offsets (a_offs / b_offs may be null: no such context).  Mixture frames
// [start_frame, T_u) are kept, and every mixture must have more than start_frame frames; frame t of x[160 s:] is
// frame t + s of x, so the kept frames are transformed from mix_offs[u] + 160 * start_frame on.  Every context must
// yield the 200 frames the towers read.
int batch_geometry(nhans_ctx* ctx, const int64_t* mix_offs, const int64_t* a_offs, const int64_t* b_offs, int U,
                   int start_frame, Geometry& g) {
  auto rel = [&](const int64_t* o, std::vector<long long>& v) {
    v.clear();
    if (o) for (int u = 0; u <= U; ++u) v.push_back(o[u] - o[0]);
  };
  auto short_ctx = [](const std::vector<long long>& o, int u) { return !o.empty() && frames_of(o[u + 1] - o[u]) < kCtxFrames; };
  g.U = U;
  rel(mix_offs, g.mix_offs);
  rel(a_offs, g.a_offs);
  rel(b_offs, g.b_offs);
  g.frame_offs.assign(U + 1, 0);
  g.out_offs.assign(U + 1, 0);
  g.ctx_frame_offs.resize(U + 1);
  g.max_frames = 0;
  const int skip = std::max(start_frame, 0);
  for (int u = 0; u < U; ++u) {
    const int T = frames_of(g.mix_offs[u + 1] - g.mix_offs[u]);
    if (start_frame != kWholeClips && T <= start_frame)
      return fail(ctx, NHANS_ERR_ARG, "utterance " + std::to_string(u) + " has " + std::to_string(T) + " <= start_frame frames");
    if (short_ctx(g.b_offs, u) || short_ctx(g.a_offs, u))
      return fail(ctx, NHANS_ERR_CONTEXT_TOO_SHORT,
                  "context clip of utterance " + std::to_string(u) + " yields fewer than 200 STFT frames (needs >= 32240 samples)");
    const int kept = T - skip;
    g.max_frames = std::max(g.max_frames, kept);
    g.frame_offs[u + 1] = g.frame_offs[u] + kept;
    g.out_offs[u + 1] = g.out_offs[u] + out_len(kept);
  }
  for (int u = 0; u < U; ++u) g.mix_offs[u] += 160LL * skip;
  for (int u = 0; u <= U; ++u) g.ctx_frame_offs[u] = (long long)u * kCtxFrames;
  g.total_frames = g.frame_offs[U];
  g.total_out = g.out_offs[U];
  return 0;
}

int need_weights(nhans_ctx* ctx) {
  if (!ctx->main_net.ready || !ctx->tower.ready) return fail(ctx, NHANS_ERR_STATE, "nhans_load_weights has not been called");
  return 0;
}

// ctx_a comes with its offsets, and only the selective-noise variant may leave it out (Silent.wav conditions instead).
int check_contexts(nhans_ctx* ctx, const void* ctx_a, const int64_t* a_offs) {
  if (ctx_a && !a_offs) return fail(ctx, NHANS_ERR_ARG, "ctx_a given without offsets");
  if (!ctx_a && ctx->variant != NHANS_VARIANT_SELECTIVE_NOISE)
    return fail(ctx, NHANS_ERR_ARG, "the separator needs both context recordings");
  return 0;
}

// Copies the n samples of x from offs[0] on into d on `stream`.
template <class T>
int copy_clips(nhans_ctx* ctx, DBuf& d, const T* x, const int64_t* offs, long long n, cudaStream_t stream) {
  CK(d.ensure(n * sizeof(T) + 32));
  CK(cudaMemcpyAsync(d.p, x + offs[0], n * sizeof(T), cudaMemcpyHostToDevice, stream));
  return 0;
}

// STFT of int16 PCM (scaled by 1 / (peak + 1e-6) on the fly) or of float samples (as they are)
cudaError_t launch_stft_of(cudaStream_t s, const int16_t* pcm, const long long* offs, const long long* frame_offs, int U,
                           const int* peak, int max_frames, float* logmag, float* phase, bool phasor) {
  return launch_stft(s, pcm, offs, frame_offs, U, peak, max_frames, logmag, phase, phasor);
}
cudaError_t launch_stft_of(cudaStream_t s, const float* x, const long long* offs, const long long* frame_offs, int U,
                           const int*, int max_frames, float* logmag, float* phase, bool phasor) {
  return launch_stft_f32(s, x, offs, frame_offs, U, max_frames, logmag, phase, phasor);
}

// Copies a batch's clips (int16 or float samples) and its offset arrays into `io` on `stream`.  ctx_a may be null.
template <class T>
int stage_batch(nhans_ctx* ctx, IoSlot& io, const Geometry& g, const T* mix, const int64_t* mix_offs, const T* ctx_a,
                const int64_t* a_offs, const T* ctx_b, const int64_t* b_offs, cudaStream_t stream) {
  const int U = g.U;
  int rc;
  if ((rc = copy_clips(ctx, io.mix, mix, mix_offs, g.mix_offs[U], stream))) return rc;
  if ((rc = copy_clips(ctx, io.b, ctx_b, b_offs, g.b_offs[U], stream))) return rc;
  if (ctx_a && (rc = copy_clips(ctx, io.a, ctx_a, a_offs, g.a_offs[U], stream))) return rc;
  Staging& s = io.staging.reset();
  const size_t mo = s.add(g.mix_offs), ao = s.add(g.a_offs), bo = s.add(g.b_offs), fo = s.add(g.frame_offs),
               oo = s.add(g.out_offs), co = s.add(g.ctx_frame_offs);
  CK(s.upload(stream));
  io.mix_offs = s.ptr<long long>(mo); io.a_offs = ctx_a ? s.ptr<long long>(ao) : nullptr; io.b_offs = s.ptr<long long>(bo);
  io.frame_offs = s.ptr<long long>(fo); io.out_offs = s.ptr<long long>(oo); io.ctx_frame_offs = s.ptr<long long>(co);
  return 0;
}

// Conditioning rows of U context pairs on the compute stream (a2-a4 of SN/apply.py:359-387 for the first 200 frames
// of each context, the embedding towers, the conditioning table) -> c.cond [U][n_cols].  a = null: the cached
// Silent.wav embedding (ensure_silent must have run).
template <class T>
int run_conditioning(nhans_ctx* ctx, CondBufs& c, const T* a, const long long* d_a_offs, const T* b, const long long* d_b_offs,
                     const long long* d_ctx_frame_offs, int U) {
  constexpr bool pcm = std::is_same<T, int16_t>::value;
  const size_t cbytes = (size_t)U * kCtxFrames * kBins * 4;
  const int n_cols = ctx->main_net.plan.cond.n_cols;
  cudaStream_t st = ctx->stream;
  CK(c.ctxlm_b.ensure(cbytes));
  CK(c.emb_b.ensure((size_t)U * 512 * 4));
  CK(c.cond.ensure((size_t)U * n_cols * 4));
  if (a) {
    CK(c.ctxlm_a.ensure(cbytes));
    CK(c.emb_a.ensure((size_t)U * 512 * 4));
  }
  if (pcm) {
    CK(c.peak_a.ensure(sizeof(int) * U));
    CK(c.peak_b.ensure(sizeof(int) * U));
    LAUNCH(launch_peaks(st, reinterpret_cast<const int16_t*>(b), d_b_offs, U, c.peak_b.as<int>()));
  }
  {
    ProfScope ps(ctx, 4, 0, 0);
    LAUNCH(launch_stft_of(st, b, d_b_offs, d_ctx_frame_offs, U, c.peak_b.as<int>(), kCtxFrames, c.ctxlm_b.as<float>(), nullptr, false));
  }
  const float* emb_a = ctx->silent_emb.as<float>();
  int stride_a = 0;
  int rc;
  if (a) {
    if (pcm) LAUNCH(launch_peaks(st, reinterpret_cast<const int16_t*>(a), d_a_offs, U, c.peak_a.as<int>()));
    {
      ProfScope ps(ctx, 4, 0, 0);
      LAUNCH(launch_stft_of(st, a, d_a_offs, d_ctx_frame_offs, U, c.peak_a.as<int>(), kCtxFrames, c.ctxlm_a.as<float>(), nullptr, false));
    }
    // embedding towers: once per distinct context clip (SURVEY.md F6), not once per window
    if ((rc = run_tower(ctx, c.ctxlm_a.as<float>(), U, c.emb_a.as<float>()))) return rc;
    emb_a = c.emb_a.as<float>();
    stride_a = 512;
  }
  if ((rc = run_tower(ctx, c.ctxlm_b.as<float>(), U, c.emb_b.as<float>()))) return rc;
  ProfScope ps(ctx, 4, 0, 0);
  LAUNCH(launch_cond_table(st, emb_a, stride_a, c.emb_b.as<float>(), 512, U, ctx->main_net.Pa, ctx->main_net.Pb, ctx->main_net.c,
                           n_cols, c.cond.as<float>()));
  return 0;
}

// The fused path up to the inverse STFT, on the compute stream, for the batch staged in `io` (int16 or float samples):
// a2-a4 for the mixture and the first 200 frames of each context (SN/apply.py:359-387), the embedding towers, the
// conditioning table and the mask network.  Leaves batch.logmag / phase / den filled.
template <class T>
int run_fused(nhans_ctx* ctx, IoSlot& io) {
  constexpr bool pcm = std::is_same<T, int16_t>::value;
  Batch& b = ctx->batch;
  const Geometry& g = b.geo;
  const int U = g.U;
  const size_t sbytes = (size_t)g.total_frames * kBins * 4;
  cudaStream_t st = ctx->stream;
  CK(b.peak_mix.ensure(sizeof(int) * U));
  CK(b.logmag.ensure(sbytes + 4));
  CK(b.phase.ensure(2 * sbytes + 8));          // unit phasors (float2 per bin) between the two transforms
  CK(b.den.ensure(sbytes + 4));
  if (pcm)
    LAUNCH(launch_peaks(st, io.mix.as<int16_t>(), io.mix_offs, U, b.peak_mix.as<int>()));
  else
    CK(cudaMemsetAsync(b.peak_mix.p, 0, sizeof(int) * U, st));     // the inverse STFT reads it; no int16 output here
  {
    ProfScope ps(ctx, 1, 0, (double)sizeof(T) * g.mix_offs[U] + 3.0 * sbytes);
    LAUNCH(launch_stft_of(st, io.mix.as<T>(), io.mix_offs, io.frame_offs, U, b.peak_mix.as<int>(), g.max_frames,
                          b.logmag.as<float>(), b.phase.as<float>(), true));
  }
  int rc;
  if ((rc = run_conditioning(ctx, b.cb, b.has_a ? io.a.as<T>() : nullptr, io.a_offs, io.b.as<T>(), io.b_offs, io.ctx_frame_offs, U)))
    return rc;
  return run_masknet(ctx, b.logmag.as<float>(), io.frame_offs, g.frame_offs.data(), io.frame_offs, g.frame_offs.data(), nullptr,
                     nullptr, U, b.cb.cond.as<float>(), b.den.as<float>());
}

// Inverse STFT on the compute stream of the batch staged in `io`: `spec` (batch.den or batch.logmag) with the
// phasors of batch.phase -> out_f32 / out_i16 (either may be null).
int batch_istft(nhans_ctx* ctx, const IoSlot& io, const DBuf& spec, float* out_f32, int16_t* out_i16) {
  const Batch& b = ctx->batch;
  const Geometry& g = b.geo;
  // spectrum + phasors read, samples written
  ProfScope ps(ctx, 2, 0, 3.0 * 4 * kBins * g.total_frames + ((out_f32 ? 4.0 : 0.0) + (out_i16 ? 2.0 : 0.0)) * g.total_out);
  LAUNCH(launch_istft(ctx->stream, spec.as<float>(), b.phase.as<float>(), io.frame_offs, io.out_offs, g.U, b.peak_mix.as<int>(),
                      g.max_frames, out_f32, out_i16, true));
  return 0;
}

// nhans_stft / nhans_stft_f32
template <class T>
int stft_entry(nhans_ctx* ctx, const T* x, const int64_t* offs, int U, float* logmag, float* phase, int64_t* frame_offs,
               int32_t* peak) {
  constexpr bool pcm = std::is_same<T, int16_t>::value;
  if (!ctx || !x || !offs || !frame_offs || U <= 0) return fail(ctx, NHANS_ERR_ARG, "bad arguments");
  CK(cudaSetDevice(ctx->device));
  Geometry g;
  int rc;
  if ((rc = batch_geometry(ctx, offs, nullptr, nullptr, U, kWholeClips, g))) return rc;
  std::copy(g.frame_offs.begin(), g.frame_offs.end(), frame_offs);
  if (!logmag && !phase && !peak) return NHANS_OK;
  const long long total = g.mix_offs[U];
  if ((rc = copy_clips(ctx, ctx->tmp[0], x, offs, total, ctx->stream))) return rc;
  Staging& s = ctx->staging.reset();
  const size_t mo = s.add(g.mix_offs), fo = s.add(g.frame_offs);
  CK(s.upload(ctx->stream));
  const size_t sbytes = (size_t)g.total_frames * kBins * 4;
  CK(ctx->tmp[4].ensure(sbytes + 4));
  CK(ctx->tmp[5].ensure(sbytes + 4));
  if (pcm) {
    CK(ctx->tmp[3].ensure(sizeof(int) * U));
    LAUNCH(launch_peaks(ctx->stream, ctx->tmp[0].as<int16_t>(), s.ptr<long long>(mo), U, ctx->tmp[3].as<int>()));
  }
  {
    ProfScope ps(ctx, 1, 0, (double)sizeof(T) * total + 2.0 * sbytes);
    LAUNCH(launch_stft_of(ctx->stream, ctx->tmp[0].as<T>(), s.ptr<long long>(mo), s.ptr<long long>(fo), U, ctx->tmp[3].as<int>(),
                          g.max_frames, ctx->tmp[4].as<float>(), ctx->tmp[5].as<float>(), false));
  }
  if (logmag) CK(cudaMemcpyAsync(logmag, ctx->tmp[4].p, sbytes, cudaMemcpyDeviceToHost, ctx->stream));
  if (phase) CK(cudaMemcpyAsync(phase, ctx->tmp[5].p, sbytes, cudaMemcpyDeviceToHost, ctx->stream));
  if (peak) CK(cudaMemcpyAsync(peak, ctx->tmp[3].p, sizeof(int) * U, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return NHANS_OK;
}

// ---- streaming -----------------------------------------------------------------------------------
constexpr int kHalfWin = kWinFrames / 2;      // 17: frames a window reaches on either side of its centre

// Windows of a stream that has F frames: all of them after the final step, else those whose 17 right-hand frames
// exist.  Output hop h needs denoised frames h - 2 .. h, so a stream that has windows [0, b) has emitted hops [0, b),
// and after its final step the whole (F - 1) * 160 + 400 samples of the batch path.
long long stream_windows(int F, bool final) { return final ? F : std::max(0, F - kHalfWin); }
long long stream_emitted(int F, bool final) { return final ? out_len(F) : 160LL * stream_windows(F, false); }

// A slot of the state pool for each of n new streams; the pool grows (keeping its contents) when none is free.
int alloc_slots(nhans_ctx* ctx, int n, std::vector<int>& slots) {
  Streams& S = ctx->streams;
  if ((int)S.free_slots.size() < n) {
    const int n_cols = ctx->main_net.plan.cond.n_cols;
    const long long stride = (kSlotCond + n_cols + 3) / 4 * 4;
    const int want = std::max({S.n_slots * 2, S.n_slots + n - (int)S.free_slots.size(), 16});
    DBuf grown;
    CK(grown.ensure((size_t)want * stride * 4));
    if (S.n_slots) CK(cudaMemcpyAsync(grown.p, S.pool.p, (size_t)S.n_slots * stride * 4, cudaMemcpyDeviceToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    S.pool = std::move(grown);
    S.slot_stride = stride;
    for (int i = want - 1; i >= S.n_slots; --i) S.free_slots.push_back(i);
    S.n_slots = want;
  }
  slots.resize(n);
  for (int i = 0; i < n; ++i) {
    slots[i] = S.free_slots.back();
    S.free_slots.pop_back();
  }
  return 0;
}

// The streams of a step must be open, distinct and not finalised.
int check_stream_ids(nhans_ctx* ctx, int n, const int* ids, bool for_step) {
  std::unordered_set<int> seen;
  for (int i = 0; i < n; ++i) {
    auto it = ctx->streams.rec.find(ids[i]);
    if (it == ctx->streams.rec.end()) return fail(ctx, NHANS_ERR_ARG, "stream id " + std::to_string(ids[i]) + " is not open");
    if (!seen.insert(ids[i]).second) return fail(ctx, NHANS_ERR_ARG, "stream id " + std::to_string(ids[i]) + " appears twice");
    if (for_step && it->second.final)
      return fail(ctx, NHANS_ERR_ARG, "stream id " + std::to_string(ids[i]) + " has had its final step");
  }
  return 0;
}

// The post-mix outputs of nhans_stream_step_post (null: a plain step).
struct PostOut {
  const float* compensate;          // [n] or null (0)
  float *mixed, *removed, *comp, *snr_est;
};

// nhans_stream_step and, with `post`, nhans_stream_step_post.
int stream_step(nhans_ctx* ctx, int n, const int* ids, const int16_t* pcm, const int64_t* offs, const int* final, int16_t* out_i16,
                float* out_f32, int64_t* out_offs, const PostOut* post) {
  if (!ctx || n < 0 || n > 65535 || !out_offs || (n > 0 && (!ids || !offs))) return fail(ctx, NHANS_ERR_ARG, "bad arguments");
  out_offs[0] = 0;
  if (n == 0) return NHANS_OK;
  for (int i = 0; i < n; ++i)
    if (offs[i + 1] < offs[i]) return fail(ctx, NHANS_ERR_ARG, "chunk offsets must not decrease");
  if (offs[n] > offs[0] && !pcm) return fail(ctx, NHANS_ERR_ARG, "bad arguments");
  int rc;
  if ((rc = need_weights(ctx))) return rc;
  if ((rc = check_stream_ids(ctx, n, ids, true))) return rc;
  CK(cudaSetDevice(ctx->device));
  Streams& S = ctx->streams;
  // Geometry of the step (kernels.h StreamStepDev).  Stream i has F0 frames before the step and F1 after it; its windows
  // [a, b) run now.  It stores frames [cs, F1), cs = a - 17 (or 0): the carry = F0 - cs frames of its slot, then the new
  // ones.  Its denoised frames a - dc .. b - 1 go through the inverse STFT.
  // offsets [n + 1] of the staged samples, new frames, segment rows, windows and emitted samples; the rest is per stream
  std::vector<long long> pcm_o(n + 1, 0), new_o(n + 1, 0), seg_o(n + 1, 0), win_o(n + 1, 0), out_o(n + 1, 0);
  std::vector<int> slot(n), carry(n), left(n), den_carry(n), keep(n), den_keep(n), peak(n);
  int max_new = 0, max_rows = 0, max_wins = 0, max_keep = 0;
  long long max_out = 0;
  std::vector<int> F1s(n);
  for (int i = 0; i < n; ++i) {
    const StreamRec& r = S.rec.at(ids[i]);
    const bool fin = final && final[i];
    const long long len = offs[i + 1] - offs[i], N1 = r.n + len;
    const int F0 = frames_of(r.n), F1 = frames_of(N1);
    const long long a = stream_windows(F0, false), b = std::max(a, stream_windows(F1, fin));
    const long long cs = std::max(0LL, a - kHalfWin);
    slot[i] = r.slot;
    peak[i] = r.peak;
    carry[i] = (int)(F0 - cs);
    left[i] = (int)(a - cs);
    den_carry[i] = (int)std::min(a, 2LL);
    keep[i] = (int)(std::max(0LL, b - kHalfWin) - cs);
    den_keep[i] = (int)std::min(b, 2LL);
    F1s[i] = F1;
    pcm_o[i + 1] = pcm_o[i] + (long long)r.tail.size() + len;
    new_o[i + 1] = new_o[i] + (F1 - F0);
    seg_o[i + 1] = seg_o[i] + (F1 - cs);
    win_o[i + 1] = win_o[i] + (b - a);
    out_o[i + 1] = out_o[i] + stream_emitted(F1, fin) - stream_emitted(F0, false);
    max_new = std::max(max_new, F1 - F0);
    max_rows = std::max<long long>(max_rows, F1 - cs);
    max_wins = std::max<long long>(max_wins, b - a);
    max_keep = std::max<long long>(max_keep, F1 - cs - keep[i]);
    max_out = std::max(max_out, out_o[i + 1] - out_o[i]);
  }
  const int n_cols = ctx->main_net.plan.cond.n_cols;
  const long long n_new = new_o[n], n_seg = seg_o[n], n_win = win_o[n], n_out = out_o[n];
  if (n_seg > 0x7fffffffLL) return fail(ctx, NHANS_ERR_ARG, "too many frames in one step");
  // staging: each stream's unframed tail, then its chunk
  std::vector<int16_t> staged((size_t)pcm_o[n]);
  for (int i = 0; i < n; ++i) {
    const StreamRec& r = S.rec.at(ids[i]);
    std::copy(r.tail.begin(), r.tail.end(), staged.begin() + pcm_o[i]);
    if (offs[i + 1] > offs[i]) std::copy(pcm + offs[i], pcm + offs[i + 1], staged.begin() + pcm_o[i] + r.tail.size());
  }
  std::vector<float> factor;        // post step: compensation factor of each stream
  if (post)
    for (int i = 0; i < n; ++i) {
      const float c = post->compensate ? post->compensate[i] : 0.f;
      factor.push_back(std::isfinite(c) ? c : 0.f);       // the batch rule (compensate_kernel)
    }
  cudaStream_t st = ctx->stream;
  Staging& sg = ctx->staging.reset();
  const size_t o_pcm = sg.add(pcm_o), o_new = sg.add(new_o), o_seg = sg.add(seg_o), o_win = sg.add(win_o), o_out = sg.add(out_o);
  const size_t o_slot = sg.add(slot), o_carry = sg.add(carry), o_left = sg.add(left), o_den_carry = sg.add(den_carry),
               o_keep = sg.add(keep), o_den_keep = sg.add(den_keep), o_peak = sg.add(peak), o_factor = sg.add(factor);
  CK(sg.upload(st));
  CK(S.pcm.ensure(staged.size() * 2 + 32));
  CK(S.new_lm.ensure((size_t)n_new * kBins * 4 + 4));
  CK(S.new_ph.ensure((size_t)n_new * kBins * 8 + 8));
  CK(S.seg_lm.ensure((size_t)n_seg * kBins * 4 + 4));
  CK(S.seg_ph.ensure((size_t)n_seg * kBins * 8 + 8));
  CK(S.den_seg.ensure((size_t)n_seg * kBins * 4 + 4));
  CK(S.den_win.ensure((size_t)n_win * kBins * 4 + 4));
  CK(S.cond.ensure((size_t)n * n_cols * 4));
  CK(S.out_f32.ensure((size_t)n_out * 4 + 16));
  CK(S.out_i16.ensure((size_t)n_out * 2 + 16));
  if (!staged.empty()) CK(cudaMemcpyAsync(S.pcm.p, staged.data(), staged.size() * 2, cudaMemcpyHostToDevice, st));
  StreamStepDev p;
  p.n = n;
  p.seg_offs = sg.ptr<long long>(o_seg); p.new_offs = sg.ptr<long long>(o_new); p.win_offs = sg.ptr<long long>(o_win);
  p.out_offs = sg.ptr<long long>(o_out);
  p.slot = sg.ptr<int>(o_slot); p.carry = sg.ptr<int>(o_carry); p.left = sg.ptr<int>(o_left); p.den_carry = sg.ptr<int>(o_den_carry);
  p.keep = sg.ptr<int>(o_keep); p.den_keep = sg.ptr<int>(o_den_keep); p.peak = sg.ptr<int>(o_peak);
  p.pool = S.pool.as<float>(); p.slot_stride = S.slot_stride; p.n_cols = n_cols;
  p.new_lm = S.new_lm.as<float>(); p.new_ph = S.new_ph.as<float>(); p.den_win = S.den_win.as<float>();
  p.seg_lm = S.seg_lm.as<float>(); p.seg_ph = S.seg_ph.as<float>(); p.den_seg = S.den_seg.as<float>(); p.cond = S.cond.as<float>();
  {
    ProfScope ps(ctx, 1, 0, 2.0 * pcm_o[n] + 12.0 * n_new * kBins);
    LAUNCH(launch_stft(st, S.pcm.as<int16_t>(), sg.ptr<long long>(o_pcm), p.new_offs, n, p.peak, max_new, S.new_lm.as<float>(),
                       S.new_ph.as<float>(), true));
  }
  LAUNCH(launch_stream_assemble(st, p, max_rows));
  if (n_win > 0) {
    // (no pass when no window became computable)
    if ((rc = run_masknet(ctx, p.seg_lm, p.seg_offs, seg_o.data(), p.win_offs, win_o.data(), p.left, left.data(), n, p.cond,
                          S.den_win.as<float>())))
      return rc;
    LAUNCH(launch_stream_den(st, p, max_wins));
  }
  // the post step always runs its inverse STFT: the running snr_est covers every sample it emits, wanted or not
  std::vector<double> sums(post ? 2 * n : 0);
  if (post) {
    CK(S.sums.ensure(sizeof(double) * 2 * n));
    CK(S.mixed.ensure((size_t)n_out * 4 + 16));
    CK(S.removed.ensure((size_t)n_out * 4 + 16));
    CK(S.comp.ensure((size_t)n_out * 4 + 16));
    ProfScope ps(ctx, 2, 0, 24.0 * n_win * kBins + 18.0 * n_out);
    LAUNCH(launch_istft_stream_post(st, p, (int)max_out, sg.ptr<float>(o_factor), out_f32 ? S.out_f32.as<float>() : nullptr,
                                    out_i16 ? S.out_i16.as<int16_t>() : nullptr, post->mixed ? S.mixed.as<float>() : nullptr,
                                    post->removed ? S.removed.as<float>() : nullptr, post->comp ? S.comp.as<float>() : nullptr,
                                    S.sums.as<double>()));
  } else if (out_f32 || out_i16) {
    ProfScope ps(ctx, 2, 0, 12.0 * n_win * kBins + 6.0 * n_out);
    LAUNCH(launch_istft_stream(st, p, (int)max_out, out_f32 ? S.out_f32.as<float>() : nullptr,
                               out_i16 ? S.out_i16.as<int16_t>() : nullptr));
  }
  LAUNCH(launch_stream_save(st, p, max_keep));
  if (out_f32 && n_out) CK(cudaMemcpyAsync(out_f32, S.out_f32.p, n_out * 4, cudaMemcpyDeviceToHost, st));
  if (out_i16 && n_out) CK(cudaMemcpyAsync(out_i16, S.out_i16.p, n_out * 2, cudaMemcpyDeviceToHost, st));
  if (post) {
    if (post->mixed && n_out) CK(cudaMemcpyAsync(post->mixed, S.mixed.p, n_out * 4, cudaMemcpyDeviceToHost, st));
    if (post->removed && n_out) CK(cudaMemcpyAsync(post->removed, S.removed.p, n_out * 4, cudaMemcpyDeviceToHost, st));
    if (post->comp && n_out) CK(cudaMemcpyAsync(post->comp, S.comp.p, n_out * 4, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(sums.data(), S.sums.p, sizeof(double) * 2 * n, cudaMemcpyDeviceToHost, st));
  }
  if ((rc = finish(ctx, cudaStreamSynchronize(st)))) return rc;
  for (int i = 0; i < n; ++i) {
    StreamRec& r = S.rec.at(ids[i]);
    const long long F0 = frames_of(r.n);
    // the next frame starts at sample 160 F1: keep the staged samples from there on
    const long long from = 160LL * (F1s[i] - F0);
    r.tail.assign(staged.begin() + pcm_o[i] + from, staged.begin() + pcm_o[i + 1]);
    r.n += offs[i + 1] - offs[i];
    r.final = final && final[i];
    out_offs[i + 1] = out_o[i + 1];
    if (post) {
      r.e_den += sums[2 * i];
      r.e_rem += sums[2 * i + 1];
      // both means share the sample count, so snr_est is the ratio of the sums (compensate_kernel)
      if (post->snr_est) post->snr_est[i] = (float)(r.e_rem > 0 ? r.e_den / r.e_rem : INFINITY);
    }
  }
  return NHANS_OK;
}

}  // namespace

// ================================================================================================
// C ABI
// ================================================================================================
extern "C" {

const char* nhans_last_error(const nhans_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int nhans_create(int device, int variant, int win_capacity, int row_capacity, nhans_ctx** out) {
  if (!out) return NHANS_ERR_ARG;
  *out = nullptr;
  if (variant != 0 && variant != 1) { g_create_error = "variant must be 0 or 1"; return NHANS_ERR_ARG; }
  int n_dev = 0;
  cudaError_t e = cudaGetDeviceCount(&n_dev);
  if (e != cudaSuccess || n_dev <= 0) {
    g_create_error = std::string("no usable CUDA device (") + cudaGetErrorString(e) + "); this library has no CPU fallback";
    return NHANS_ERR_CUDA;
  }
  if (device < 0 || device >= n_dev) { g_create_error = "device index out of range"; return NHANS_ERR_ARG; }
  if ((e = cudaSetDevice(device)) != cudaSuccess) { g_create_error = cudaGetErrorString(e); return NHANS_ERR_CUDA; }
  cudaDeviceProp prop;
  if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) { g_create_error = cudaGetErrorString(e); return NHANS_ERR_CUDA; }
  if (prop.major != 10) {
    g_create_error = "device is sm_" + std::to_string(prop.major) + std::to_string(prop.minor) + "; this library is built for sm_100a (B200) only";
    return NHANS_ERR_CUDA;
  }
  std::unique_ptr<nhans_ctx> c(new nhans_ctx);
  nhans_ctx* ctx = c.get();
  ctx->device = device;
  ctx->variant = variant;
  if (win_capacity > 0) ctx->win_cap = win_capacity;
  if (row_capacity > 0) ctx->row_cap = row_capacity;
  if (const char* dbg = getenv("NHANS_DEBUG_TIMELINE")) ctx->timeline = atoi(dbg) != 0;
  if (const char* dbg = getenv("NHANS_NO_WALK")) ctx->use_walk = atoi(dbg) == 0;
  if (const char* dbg = getenv("NHANS_NO_GEN")) ctx->use_gen = atoi(dbg) == 0;
  if (const char* dbg = getenv("NHANS_DEBUG_STATS")) {
    if (atoi(dbg) && cudaMalloc((void**)&ctx->debug_stats, 128 * 8 * 8) == cudaSuccess) cudaMemset(ctx->debug_stats, 0, 128 * 8 * 8);
  }
  ctx->n_sm = prop.multiProcessorCount;
  auto bail = [&](const std::string& m) { g_create_error = m; return NHANS_ERR_CUDA; };
  if ((e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking)) != cudaSuccess) return bail(cudaGetErrorString(e));
  if ((e = cudaStreamCreateWithFlags(&ctx->h2d_stream, cudaStreamNonBlocking)) != cudaSuccess) return bail(cudaGetErrorString(e));
  if ((e = cudaStreamCreateWithFlags(&ctx->d2h_stream, cudaStreamNonBlocking)) != cudaSuccess) return bail(cudaGetErrorString(e));
  for (IoSlot& io : ctx->batch.io)
    for (cudaEvent_t* ev : {&io.uploaded, &io.consumed, &io.drained})
      if ((e = cudaEventCreateWithFlags(ev, cudaEventDisableTiming)) != cudaSuccess) return bail(cudaGetErrorString(e));
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if ((e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres)) != cudaSuccess || !fn)
    return bail("cuTensorMapEncodeTiled is unavailable");
  ctx->encode = reinterpret_cast<EncodeTiledFn>(fn);
  if ((e = cudaHostAlloc((void**)&ctx->err_flag_host, sizeof(int), cudaHostAllocMapped)) != cudaSuccess) return bail(cudaGetErrorString(e));
  *ctx->err_flag_host = 0;
  if ((e = cudaHostGetDevicePointer((void**)&ctx->err_flag_dev, ctx->err_flag_host, 0)) != cudaSuccess) return bail(cudaGetErrorString(e));
  if ((e = dsp_init_tables()) != cudaSuccess) return bail(std::string("dsp_init_tables: ") + cudaGetErrorString(e));
  for (auto& ev : ctx->events) cudaEventCreate(&ev);
  *out = c.release();
  return NHANS_OK;
}

void nhans_destroy(nhans_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  for (cudaStream_t s : {ctx->stream, ctx->h2d_stream, ctx->d2h_stream}) cudaStreamSynchronize(s);
  delete ctx;
}

int nhans_load_weights(nhans_ctx* ctx, const char* const* names, const int64_t* sizes, const float* const* data, int n) {
  if (!ctx || !names || !sizes || !data || n <= 0) return fail(ctx, NHANS_ERR_ARG, "bad arguments");
  CK(cudaSetDevice(ctx->device));
  WeightMap w;
  for (int i = 0; i < n; ++i) w[names[i]] = std::vector<float>(data[i], data[i] + sizes[i]);
  ctx->main_net = NetDev{};
  ctx->tower = NetDev{};
  ctx->silent_ready = false;
  // open streams end, since their conditioning rows belong to the old weights; ids go on counting, so that an id from
  // before the reload never names a new stream
  const int next_id = ctx->streams.next_id;
  ctx->streams = Streams{};
  ctx->streams.next_id = next_id;
  try {
    ctx->main_net.plan = build_main_plan(w, ctx->variant, ctx->win_cap);
    ctx->tower.plan = build_tower_plan(w, ctx->row_cap);
  } catch (const std::exception& ex) {
    return fail(ctx, NHANS_ERR_ARG, std::string("weights rejected: ") + ex.what());
  }
  int rc;
  if ((rc = realise_net(ctx, ctx->main_net))) return rc;
  if ((rc = realise_net(ctx, ctx->tower))) return rc;
  // the packed host copies are no longer needed
  for (NetDev* nd : {&ctx->main_net, &ctx->tower})
    for (auto& L : nd->plan.gemm) {
      if (L.subnormal_frac > 0.01)
        fprintf(stderr, "nhans: warning: %.1f %% of the fp16 weights of layer %s are subnormal (reduced precision)\n",
                100.0 * L.subnormal_frac, L.name.c_str());
      std::vector<uint16_t>().swap(L.w);
    }
  if (ctx->err_flag_host) *ctx->err_flag_host = 0;
  return NHANS_OK;
}

int nhans_output_offsets(const int64_t* mix_offs, int U, int64_t* out_offs) {
  if (!mix_offs || !out_offs || U < 0) return NHANS_ERR_ARG;
  Geometry g;
  batch_geometry(nullptr, mix_offs, nullptr, nullptr, U, kWholeClips, g);     // checks nothing without contexts
  std::copy(g.out_offs.begin(), g.out_offs.end(), out_offs);
  return NHANS_OK;
}

int nhans_normalise(nhans_ctx* ctx, const int16_t* pcm, const int64_t* offs, int U, int trim, float* out, int64_t* out_offs) {
  if (!ctx || !pcm || !offs || !out || !out_offs || U <= 0) return fail(ctx, NHANS_ERR_ARG, "bad arguments");
  CK(cudaSetDevice(ctx->device));
  std::vector<long long> rel(U + 1), oo(U + 1, 0);      // input offsets relative to offs[0], output offsets
  for (int u = 0; u <= U; ++u) rel[u] = offs[u] - offs[0];
  for (int u = 0; u < U; ++u) {
    long long n = rel[u + 1] - rel[u];
    if (trim && n >= 400) n -= (n - 400) % 160;
    oo[u + 1] = oo[u] + n;
  }
  int rc;
  if ((rc = copy_clips(ctx, ctx->tmp[0], pcm, offs, rel[U], ctx->stream))) return rc;
  Staging& s = ctx->staging.reset();
  const size_t ro = s.add(rel), o_oo = s.add(oo);
  CK(s.upload(ctx->stream));
  CK(ctx->tmp[3].ensure(sizeof(int) * U));
  CK(ctx->tmp[4].ensure(oo[U] * 4 + 4));
  LAUNCH(launch_peaks(ctx->stream, ctx->tmp[0].as<int16_t>(), s.ptr<long long>(ro), U, ctx->tmp[3].as<int>()));
  LAUNCH(launch_normalise(ctx->stream, ctx->tmp[0].as<int16_t>(), s.ptr<long long>(ro), s.ptr<long long>(o_oo), U,
                          ctx->tmp[3].as<int>(), ctx->tmp[4].as<float>()));
  CK(cudaMemcpyAsync(out, ctx->tmp[4].p, oo[U] * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  for (int u = 0; u <= U; ++u) out_offs[u] = oo[u];
  return NHANS_OK;
}

int nhans_stft(nhans_ctx* ctx, const int16_t* pcm, const int64_t* offs, int U, float* logmag, float* phase,
               int64_t* frame_offs, int32_t* peak) {
  return stft_entry(ctx, pcm, offs, U, logmag, phase, frame_offs, peak);
}

int nhans_stft_f32(nhans_ctx* ctx, const float* x, const int64_t* offs, int U, float* logmag, float* phase,
                   int64_t* frame_offs) {
  return stft_entry(ctx, x, offs, U, logmag, phase, frame_offs, nullptr);
}

int nhans_eval_loss(nhans_ctx* ctx, const float* denoised, const float* target, int64_t n_frames, float* example_loss) {
  if (!ctx || !denoised || !target || !example_loss || n_frames < 0) return fail(ctx, NHANS_ERR_ARG, "bad arguments");
  if (n_frames == 0) return NHANS_OK;
  CK(cudaSetDevice(ctx->device));
  const size_t bytes = (size_t)n_frames * kBins * 4;
  CK(ctx->tmp[0].ensure(bytes));
  CK(ctx->tmp[1].ensure(bytes));
  CK(ctx->tmp[2].ensure((size_t)n_frames * 4));
  CK(cudaMemcpyAsync(ctx->tmp[0].p, denoised, bytes, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(ctx->tmp[1].p, target, bytes, cudaMemcpyHostToDevice, ctx->stream));
  {
    ProfScope ps(ctx, 4, 0, 0);
    LAUNCH(launch_eval_loss(ctx->stream, ctx->tmp[0].as<float>(), ctx->tmp[1].as<float>(), n_frames, ctx->tmp[2].as<float>()));
  }
  CK(cudaMemcpyAsync(example_loss, ctx->tmp[2].p, (size_t)n_frames * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return NHANS_OK;
}

int nhans_embed(nhans_ctx* ctx, const float* ctx_logmag, int R, float* emb) {
  if (!ctx || !ctx_logmag || !emb || R <= 0) return fail(ctx, NHANS_ERR_ARG, "bad arguments");
  CK(cudaSetDevice(ctx->device));
  int rc;
  if ((rc = need_weights(ctx))) return rc;
  const size_t in_bytes = (size_t)R * kCtxFrames * kBins * 4;
  CK(ctx->tmp[0].ensure(in_bytes));
  CK(ctx->tmp[1].ensure((size_t)R * 512 * 4));
  CK(cudaMemcpyAsync(ctx->tmp[0].p, ctx_logmag, in_bytes, cudaMemcpyHostToDevice, ctx->stream));
  if ((rc = run_tower(ctx, ctx->tmp[0].as<float>(), R, ctx->tmp[1].as<float>()))) return rc;
  CK(cudaMemcpyAsync(emb, ctx->tmp[1].p, (size_t)R * 512 * 4, cudaMemcpyDeviceToHost, ctx->stream));
  return finish(ctx, cudaStreamSynchronize(ctx->stream));
}

int nhans_masknet(nhans_ctx* ctx, const float* logmag, const int64_t* frame_offs, int U, const float* emb_a,
                  const float* emb_b, float* denoised) {
  if (!ctx || !logmag || !frame_offs || !emb_a || !emb_b || !denoised || U <= 0) return fail(ctx, NHANS_ERR_ARG, "bad arguments");
  CK(cudaSetDevice(ctx->device));
  int rc;
  if ((rc = need_weights(ctx))) return rc;
  std::vector<long long> fo(frame_offs, frame_offs + U + 1);
  const long long total = fo[U];
  const size_t sbytes = (size_t)total * kBins * 4;
  const int n_cols = ctx->main_net.plan.cond.n_cols;
  CK(ctx->tmp[0].ensure(sbytes + 4));
  CK(ctx->tmp[1].ensure(sbytes + 4));
  CK(ctx->tmp[2].ensure((size_t)U * 512 * 4));
  CK(ctx->tmp[3].ensure((size_t)U * 512 * 4));
  CK(ctx->tmp[4].ensure((size_t)U * n_cols * 4));
  Staging& s = ctx->staging.reset();
  const size_t o_fo = s.add(fo);
  CK(s.upload(ctx->stream));
  CK(cudaMemcpyAsync(ctx->tmp[0].p, logmag, sbytes, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(ctx->tmp[2].p, emb_a, (size_t)U * 512 * 4, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(ctx->tmp[3].p, emb_b, (size_t)U * 512 * 4, cudaMemcpyHostToDevice, ctx->stream));
  LAUNCH(launch_cond_table(ctx->stream, ctx->tmp[2].as<float>(), 512, ctx->tmp[3].as<float>(), 512, U, ctx->main_net.Pa,
                           ctx->main_net.Pb, ctx->main_net.c, n_cols, ctx->tmp[4].as<float>()));
  if ((rc = run_masknet(ctx, ctx->tmp[0].as<float>(), s.ptr<long long>(o_fo), fo.data(), s.ptr<long long>(o_fo), fo.data(), nullptr,
                        nullptr, U, ctx->tmp[4].as<float>(), ctx->tmp[1].as<float>())))
    return rc;
  CK(cudaMemcpyAsync(denoised, ctx->tmp[1].p, sbytes, cudaMemcpyDeviceToHost, ctx->stream));
  return finish(ctx, cudaStreamSynchronize(ctx->stream));
}

int nhans_istft(nhans_ctx* ctx, const float* logmag, const float* phase, const int64_t* frame_offs, int U,
                const int32_t* peak, float* wav_f32, int16_t* wav_i16, int64_t* out_offs) {
  if (!ctx || !logmag || !phase || !frame_offs || !out_offs || U <= 0) return fail(ctx, NHANS_ERR_ARG, "bad arguments");
  if (wav_i16 && !peak) return fail(ctx, NHANS_ERR_ARG, "int16 output needs the input peaks");
  CK(cudaSetDevice(ctx->device));
  std::vector<long long> fo(frame_offs, frame_offs + U + 1), oo(U + 1, 0);
  int max_frames = 0;
  for (int u = 0; u < U; ++u) {
    int T = (int)(fo[u + 1] - fo[u]);
    max_frames = std::max(max_frames, T);
    oo[u + 1] = oo[u] + out_len(T);
  }
  for (int u = 0; u <= U; ++u) out_offs[u] = oo[u];
  if (!wav_f32 && !wav_i16) return NHANS_OK;
  const size_t sbytes = (size_t)fo[U] * kBins * 4;
  CK(ctx->tmp[0].ensure(sbytes + 4));
  CK(ctx->tmp[1].ensure(sbytes + 4));
  CK(cudaMemcpyAsync(ctx->tmp[0].p, logmag, sbytes, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(ctx->tmp[1].p, phase, sbytes, cudaMemcpyHostToDevice, ctx->stream));
  Staging& s = ctx->staging.reset();
  const size_t o_fo = s.add(fo), o_oo = s.add(oo), o_pk = peak ? s.add(peak, U) : s.add(std::vector<int>(U, 0));
  CK(s.upload(ctx->stream));
  CK(ctx->tmp[5].ensure(oo[U] * 4 + 4));
  CK(ctx->tmp[6].ensure(oo[U] * 2 + 4));
  {
    ProfScope ps(ctx, 2, 0, 2.0 * sbytes + (wav_f32 ? 4.0 : 0.0) * oo[U] + (wav_i16 ? 2.0 : 0.0) * oo[U]);
    LAUNCH(launch_istft(ctx->stream, ctx->tmp[0].as<float>(), ctx->tmp[1].as<float>(), s.ptr<long long>(o_fo), s.ptr<long long>(o_oo),
                        U, s.ptr<int>(o_pk), max_frames, wav_f32 ? ctx->tmp[5].as<float>() : nullptr,
                        wav_i16 ? ctx->tmp[6].as<int16_t>() : nullptr));
  }
  if (wav_f32) CK(cudaMemcpyAsync(wav_f32, ctx->tmp[5].p, oo[U] * 4, cudaMemcpyDeviceToHost, ctx->stream));
  if (wav_i16) CK(cudaMemcpyAsync(wav_i16, ctx->tmp[6].p, oo[U] * 2, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return NHANS_OK;
}

int nhans_upload(nhans_ctx* ctx, const int16_t* mix, const int64_t* mix_offs, int U, const int16_t* ctx_a,
                 const int64_t* a_offs, const int16_t* ctx_b, const int64_t* b_offs) {
  if (!ctx || !mix || !mix_offs || !ctx_b || !b_offs || U <= 0) return fail(ctx, NHANS_ERR_ARG, "bad arguments");
  int rc;
  if ((rc = check_contexts(ctx, ctx_a, a_offs))) return rc;
  CK(cudaSetDevice(ctx->device));
  if ((rc = need_weights(ctx))) return rc;
  Batch& b = ctx->batch;
  b.staged = false; b.done = false;
  b.has_a = ctx_a != nullptr;
  if ((rc = batch_geometry(ctx, mix_offs, ctx_a ? a_offs : nullptr, b_offs, U, kWholeClips, b.geo))) return rc;
  // stage into the set the previous batch does NOT use; its last user (two batches ago) must have finished
  b.cur ^= 1;
  IoSlot& io = b.io[b.cur];
  cudaStream_t hs = ctx->h2d_stream;
  CK(cudaStreamWaitEvent(hs, io.consumed, 0));
  tl_mark(ctx, 0, hs);
  if ((rc = stage_batch(ctx, io, b.geo, mix, mix_offs, ctx_a, a_offs, ctx_b, b_offs, hs))) return rc;
  tl_mark(ctx, 1, hs);
  CK(cudaEventRecord(io.uploaded, hs));
  b.staged = true;
  return NHANS_OK;
}

int nhans_run(nhans_ctx* ctx) {
  if (!ctx) return NHANS_ERR_ARG;
  Batch& b = ctx->batch;
  if (!b.staged) return fail(ctx, NHANS_ERR_STATE, "nhans_upload has not staged a batch");
  CK(cudaSetDevice(ctx->device));
  int rc;
  const Geometry& g = b.geo;
  IoSlot& io = b.io[b.cur];
  CK(io.out_i16.ensure(g.total_out * 2 + 32));
  CK(io.out_f32.ensure(g.total_out * 4 + 4));
  CK(b.mixproc.ensure(g.total_out * 4 + 4));
  if (!b.has_a && (rc = ensure_silent(ctx))) return rc;

  // the inputs of this set have landed, and the outputs the set held two batches ago have reached the host
  CK(cudaStreamWaitEvent(ctx->stream, io.uploaded, 0));
  if (io.d2h_pending) CK(cudaStreamWaitEvent(ctx->stream, io.drained, 0));
  tl_mark(ctx, 2, ctx->stream);
  if ((rc = run_fused<int16_t>(ctx, io))) return rc;
  if ((rc = batch_istft(ctx, io, b.den, io.out_f32.as<float>(), io.out_i16.as<int16_t>()))) return rc;
  tl_mark(ctx, 3, ctx->stream);
  CK(cudaEventRecord(io.consumed, ctx->stream));
  b.done = true;
  return NHANS_OK;
}

int nhans_download(nhans_ctx* ctx, int16_t* out_i16, float* out_f32, float* mixproc_f32) {
  if (!ctx) return NHANS_ERR_ARG;
  Batch& b = ctx->batch;
  if (!b.done) return fail(ctx, NHANS_ERR_STATE, "nhans_run has not produced a batch");
  const Geometry& g = b.geo;
  CK(cudaSetDevice(ctx->device));
  IoSlot& io = b.io[b.cur];
  if (mixproc_f32) {
    // 'mixed_processed.wav' (SN/apply.py:457-458): iSTFT of the window centres, i.e. of the input spectrogram
    int rc;
    if ((rc = batch_istft(ctx, io, b.logmag, b.mixproc.as<float>(), nullptr))) return rc;
    CK(cudaMemcpyAsync(mixproc_f32, b.mixproc.p, g.total_out * 4, cudaMemcpyDeviceToHost, ctx->stream));
  }
  // the outputs leave on their own stream, so that the next batch can start computing meanwhile
  CK(cudaStreamWaitEvent(ctx->d2h_stream, io.consumed, 0));
  tl_mark(ctx, 4, ctx->d2h_stream);
  if (out_i16) CK(cudaMemcpyAsync(out_i16, io.out_i16.p, g.total_out * 2, cudaMemcpyDeviceToHost, ctx->d2h_stream));
  if (out_f32) CK(cudaMemcpyAsync(out_f32, io.out_f32.p, g.total_out * 4, cudaMemcpyDeviceToHost, ctx->d2h_stream));
  tl_mark(ctx, 5, ctx->d2h_stream);
  CK(cudaEventRecord(io.drained, ctx->d2h_stream));
  io.d2h_pending = true;
  return NHANS_OK;
}

int nhans_postmix(nhans_ctx* ctx, float compensate, int ac, float* mixed_f32, float* removed_f32, float* compensated_f32,
                  float* snr_est) {
  if (!ctx) return NHANS_ERR_ARG;
  Batch& b = ctx->batch;
  if (!b.done) return fail(ctx, NHANS_ERR_STATE, "nhans_run has not produced a batch");
  const Geometry& g = b.geo;
  CK(cudaSetDevice(ctx->device));
  IoSlot& io = b.io[b.cur];
  CK(b.removed.ensure(g.total_out * 4 + 4));
  CK(b.comp.ensure(g.total_out * 4 + 4));
  CK(b.sums.ensure(sizeof(double) * 2 * g.U));
  CK(b.snr.ensure(sizeof(float) * g.U));
  {
    ProfScope ps(ctx, 2, 0, 4.0 * g.total_frames * kBins * 4 + 12.0 * g.total_out);
    LAUNCH(launch_istft_post(ctx->stream, b.den.as<float>(), b.logmag.as<float>(), b.phase.as<float>(), io.frame_offs, io.out_offs,
                             g.U, g.max_frames, nullptr, b.mixproc.as<float>(), b.removed.as<float>(), b.sums.as<double>()));
  }
  {
    ProfScope ps(ctx, 4, 0, 0);
    LAUNCH(launch_compensate(ctx->stream, io.out_f32.as<float>(), b.removed.as<float>(), io.out_offs, g.U, b.sums.as<double>(),
                             compensate, ac, compensated_f32 ? b.comp.as<float>() : nullptr, b.snr.as<float>()));
  }
  if (mixed_f32) CK(cudaMemcpyAsync(mixed_f32, b.mixproc.p, g.total_out * 4, cudaMemcpyDeviceToHost, ctx->stream));
  if (removed_f32) CK(cudaMemcpyAsync(removed_f32, b.removed.p, g.total_out * 4, cudaMemcpyDeviceToHost, ctx->stream));
  if (compensated_f32) CK(cudaMemcpyAsync(compensated_f32, b.comp.p, g.total_out * 4, cudaMemcpyDeviceToHost, ctx->stream));
  if (snr_est) CK(cudaMemcpyAsync(snr_est, b.snr.p, sizeof(float) * g.U, cudaMemcpyDeviceToHost, ctx->stream));
  return NHANS_OK;
}

int nhans_enhance_batch(nhans_ctx* ctx, const int16_t* mix, const int64_t* mix_offs, int U, const int16_t* ctx_a,
                        const int64_t* a_offs, const int16_t* ctx_b, const int64_t* b_offs, int16_t* out_i16,
                        float* out_f32, float* mixproc_f32) {
  int rc;
  if ((rc = nhans_upload(ctx, mix, mix_offs, U, ctx_a, a_offs, ctx_b, b_offs))) return rc;
  if ((rc = nhans_run(ctx))) return rc;
  return nhans_download(ctx, out_i16, out_f32, mixproc_f32);
}

int nhans_enhance_f32(nhans_ctx* ctx, const float* mix, const int64_t* mix_offs, int U, const float* ctx_a, const int64_t* a_offs,
                      const float* ctx_b, const int64_t* b_offs, int start_frame, float* out_f32, float* mixproc_f32, int64_t* out_offs) {
  if (!ctx || !mix || !mix_offs || !ctx_b || !b_offs || !out_offs || U <= 0 || start_frame < 0) return fail(ctx, NHANS_ERR_ARG, "bad arguments");
  int rc;
  if ((rc = check_contexts(ctx, ctx_a, a_offs))) return rc;
  CK(cudaSetDevice(ctx->device));
  if ((rc = need_weights(ctx))) return rc;
  Geometry geo;
  if ((rc = batch_geometry(ctx, mix_offs, ctx_a ? a_offs : nullptr, b_offs, U, start_frame, geo))) return rc;
  std::copy(geo.out_offs.begin(), geo.out_offs.end(), out_offs);
  if (!out_f32 && !mixproc_f32) return NHANS_OK;
  // the shared spectra / embedding buffers are about to be reused: nothing of an earlier batch may still be running
  CK(cudaStreamSynchronize(ctx->stream));
  CK(cudaStreamSynchronize(ctx->h2d_stream));
  CK(cudaStreamSynchronize(ctx->d2h_stream));
  Batch& b = ctx->batch;
  b.done = false; b.staged = false;
  b.geo = std::move(geo);
  b.has_a = ctx_a != nullptr;
  const Geometry& g = b.geo;
  cudaStream_t st = ctx->stream;
  IoSlot& io = b.io[b.cur];
  if ((rc = stage_batch(ctx, io, g, mix, mix_offs, ctx_a, a_offs, ctx_b, b_offs, st))) return rc;
  if (!b.has_a && (rc = ensure_silent(ctx))) return rc;
  if ((rc = run_fused<float>(ctx, io))) return rc;
  CK(io.out_f32.ensure(g.total_out * 4 + 16));
  if (out_f32) {
    if ((rc = batch_istft(ctx, io, b.den, io.out_f32.as<float>(), nullptr))) return rc;
    CK(cudaMemcpyAsync(out_f32, io.out_f32.p, g.total_out * 4, cudaMemcpyDeviceToHost, st));
  }
  if (mixproc_f32) {
    CK(b.mixproc.ensure(g.total_out * 4 + 16));
    if ((rc = batch_istft(ctx, io, b.logmag, b.mixproc.as<float>(), nullptr))) return rc;
    CK(cudaMemcpyAsync(mixproc_f32, b.mixproc.p, g.total_out * 4, cudaMemcpyDeviceToHost, st));
  }
  return finish(ctx, cudaStreamSynchronize(st));
}

int nhans_sync(nhans_ctx* ctx) {
  if (!ctx) return NHANS_ERR_ARG;
  cudaSetDevice(ctx->device);
  cudaError_t e = cudaStreamSynchronize(ctx->stream);
  cudaError_t e1 = cudaStreamSynchronize(ctx->h2d_stream);
  cudaError_t e2 = cudaStreamSynchronize(ctx->d2h_stream);
  for (IoSlot& io : ctx->batch.io) io.d2h_pending = false;
  if (int rc = finish(ctx, e)) return rc;
  CK(e1);
  CK(e2);
  return NHANS_OK;
}

int nhans_sync_previous(nhans_ctx* ctx) {
  if (!ctx) return NHANS_ERR_ARG;
  cudaSetDevice(ctx->device);
  IoSlot& io = ctx->batch.io[ctx->batch.cur ^ 1];
  if (io.d2h_pending) {
    cudaError_t e = cudaEventSynchronize(io.drained);
    io.d2h_pending = false;
    return finish(ctx, e);
  }
  return NHANS_OK;
}

int nhans_host_alloc(int64_t bytes, void** out) {
  if (!out || bytes <= 0) return NHANS_ERR_ARG;
  return cudaHostAlloc(out, (size_t)bytes, cudaHostAllocDefault) == cudaSuccess ? NHANS_OK : NHANS_ERR_CUDA;
}
void nhans_host_free(void* p) {
  if (p) cudaFreeHost(p);
}

int nhans_event_record(nhans_ctx* ctx, int slot) {
  if (!ctx || slot < 0 || slot >= 16) return NHANS_ERR_ARG;
  CK(cudaSetDevice(ctx->device));
  // the event orders after the copies of batches already enqueued, so that elapsed times cover them
  for (IoSlot& io : ctx->batch.io)
    if (io.d2h_pending) CK(cudaStreamWaitEvent(ctx->stream, io.drained, 0));
  CK(cudaEventRecord(ctx->events[slot], ctx->stream));
  return NHANS_OK;
}
int nhans_event_elapsed_ms(nhans_ctx* ctx, int a, int b, double* ms) {
  if (!ctx || !ms || a < 0 || a >= 16 || b < 0 || b >= 16) return NHANS_ERR_ARG;
  CK(cudaSetDevice(ctx->device));
  CK(cudaEventSynchronize(ctx->events[b]));
  float f = 0.f;
  CK(cudaEventElapsedTime(&f, ctx->events[a], ctx->events[b]));
  *ms = f;
  return NHANS_OK;
}

int nhans_profile_enable(nhans_ctx* ctx, int on) {
  if (!ctx) return NHANS_ERR_ARG;
  cudaSetDevice(ctx->device);
  prof_collect(ctx);
  ctx->profile = on != 0;
  return NHANS_OK;
}
int nhans_profile_get(nhans_ctx* ctx, int kind, double* stats) {
  if (!ctx || !stats || kind < 0 || kind > 5) return NHANS_ERR_ARG;
  cudaSetDevice(ctx->device);
  prof_collect(ctx);
  if (kind == 5) {
    stats[0] = ctx->launches; stats[1] = stats[2] = stats[3] = 0;
    return NHANS_OK;
  }
  for (int i = 0; i < 4; ++i) stats[i] = ctx->prof_acc[kind][i];
  return NHANS_OK;
}
int nhans_profile_reset(nhans_ctx* ctx) {
  if (!ctx) return NHANS_ERR_ARG;
  cudaSetDevice(ctx->device);
  prof_collect(ctx);
  memset(ctx->prof_acc, 0, sizeof ctx->prof_acc);
  memset(ctx->layer_acc, 0, sizeof ctx->layer_acc);
  ctx->launches = 0;
  return NHANS_OK;
}

int nhans_debug_layer_stats(nhans_ctx* ctx, int net, int layer, uint64_t* out8) {
  if (!ctx || !out8 || !ctx->debug_stats || net < 0 || net > 1 || layer < 0 || layer >= 64) return NHANS_ERR_ARG;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  return cudaMemcpy(out8, ctx->debug_stats + 8 * (net * 64 + layer), 64, cudaMemcpyDeviceToHost) == cudaSuccess ? NHANS_OK : NHANS_ERR_CUDA;
}

int nhans_profile_get_layer(nhans_ctx* ctx, int net, int layer, double* stats) {
  if (!ctx || !stats || net < 0 || net > 1 || layer < 0 || layer >= 64) return NHANS_ERR_ARG;
  cudaSetDevice(ctx->device);
  prof_collect(ctx);
  for (int i = 0; i < 4; ++i) stats[i] = ctx->layer_acc[net * 64 + layer][i];
  return NHANS_OK;
}

const char* nhans_plan_json(nhans_ctx* ctx, int net) {
  if (!ctx) return "";
  ctx->json = plan_to_json(net == 0 ? ctx->main_net.plan : ctx->tower.plan);
  return ctx->json.c_str();
}

int nhans_debug_read_buffer(nhans_ctx* ctx, int net, int buf, uint16_t* out, int64_t n_elems) {
  if (!ctx || !out) return NHANS_ERR_ARG;
  NetDev& nd = net == 0 ? ctx->main_net : ctx->tower;
  if (!nd.ready || buf < 0 || buf >= (int)nd.bufs.size()) return fail(ctx, NHANS_ERR_ARG, "no such buffer");
  const Grid& g = nd.plan.bufs[buf];
  if (n_elems > (long long)g.pixels * g.C) return fail(ctx, NHANS_ERR_ARG, "buffer is smaller than requested");
  CK(cudaSetDevice(ctx->device));
  CK(cudaStreamSynchronize(ctx->stream));
  CK(cudaMemcpy(out, nd.bufs[buf], (size_t)n_elems * 2, cudaMemcpyDeviceToHost));
  return NHANS_OK;
}

int nhans_debug_read_batch(nhans_ctx* ctx, int which, float* out, int64_t n_floats) {
  if (!ctx || !out || which < 0 || which > 2) return NHANS_ERR_ARG;
  Batch& b = ctx->batch;
  if (!b.done) return fail(ctx, NHANS_ERR_STATE, "nhans_run has not produced a batch");
  const Geometry& g = b.geo;
  const long long rows = g.total_frames * kBins;
  const long long have = which == 1 ? 2 * rows : rows;            // 1: unit phasors (float2 per bin)
  if (n_floats > have) return fail(ctx, NHANS_ERR_ARG, "the batch holds fewer values than requested");
  const DBuf& src = which == 0 ? b.logmag : (which == 1 ? b.phase : b.den);
  CK(cudaSetDevice(ctx->device));
  CK(cudaStreamSynchronize(ctx->stream));
  CK(cudaMemcpy(out, src.p, (size_t)n_floats * 4, cudaMemcpyDeviceToHost));
  return NHANS_OK;
}

int nhans_debug_timeline(nhans_ctx* ctx, double* out_ms, int max_batches) {
  if (!ctx || !out_ms || max_batches < 0) return NHANS_ERR_ARG;
  if (!ctx->timeline || !ctx->tl_origin) return 0;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  cudaStreamSynchronize(ctx->h2d_stream);
  cudaStreamSynchronize(ctx->d2h_stream);
  const int n = std::min<int>(max_batches, (int)ctx->tl.size());
  const int first = (int)ctx->tl.size() - n;
  for (int i = 0; i < n; ++i)
    for (int k = 0; k < 6; ++k) {
      float ms = -1.f;
      if (cudaEventElapsedTime(&ms, ctx->tl_origin, ctx->tl[first + i][k]) != cudaSuccess) ms = -1.f;   // never recorded
      out_ms[6 * i + k] = ms;
    }
  cudaGetLastError();
  return n;
}

int nhans_device_info(nhans_ctx* ctx, int* sm_count, int* cc_major, int* cc_minor, int64_t* mem_bytes) {
  if (!ctx) return NHANS_ERR_ARG;
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, ctx->device));
  if (sm_count) *sm_count = prop.multiProcessorCount;
  if (cc_major) *cc_major = prop.major;
  if (cc_minor) *cc_minor = prop.minor;
  if (mem_bytes) *mem_bytes = (int64_t)prop.totalGlobalMem;
  return NHANS_OK;
}

int nhans_stream_emit_len(int64_t before, int64_t after, int final, int64_t* emitted) {
  if (!emitted || before < 0 || after < before) return NHANS_ERR_ARG;
  *emitted = stream_emitted(frames_of(after), final != 0) - stream_emitted(frames_of(before), false);
  return NHANS_OK;
}

int nhans_stream_open(nhans_ctx* ctx, int n, const int16_t* ctx_a, const int64_t* a_offs, const int16_t* ctx_b,
                      const int64_t* b_offs, const int32_t* peak, int* ids) {
  if (!ctx || n <= 0 || n > 65535 || !ctx_b || !b_offs || !peak || !ids) return fail(ctx, NHANS_ERR_ARG, "bad arguments");
  int rc;
  if ((rc = check_contexts(ctx, ctx_a, a_offs))) return rc;
  for (int i = 0; i < n; ++i)
    if (peak[i] < 0) return fail(ctx, NHANS_ERR_ARG, "stream " + std::to_string(i) + " has a negative peak");
  CK(cudaSetDevice(ctx->device));
  if ((rc = need_weights(ctx))) return rc;
  // the context clips are laid out like a batch's (a mixture of zero samples per stream)
  std::vector<int64_t> no_mix(n + 1, 0);
  Geometry g;
  if ((rc = batch_geometry(ctx, no_mix.data(), ctx_a ? a_offs : nullptr, b_offs, n, kWholeClips, g))) return rc;
  Streams& S = ctx->streams;
  if (!ctx_a && (rc = ensure_silent(ctx))) return rc;
  cudaStream_t st = ctx->stream;
  if ((rc = copy_clips(ctx, S.ctx_b, ctx_b, b_offs, g.b_offs[n], st))) return rc;
  if (ctx_a && (rc = copy_clips(ctx, S.ctx_a, ctx_a, a_offs, g.a_offs[n], st))) return rc;
  Staging& sg = ctx->staging.reset();
  const size_t bo = sg.add(g.b_offs), co = sg.add(g.ctx_frame_offs), ao = sg.add(g.a_offs);
  CK(sg.upload(st));
  if ((rc = run_conditioning(ctx, S.cb, ctx_a ? S.ctx_a.as<int16_t>() : nullptr, ctx_a ? sg.ptr<long long>(ao) : nullptr,
                             S.ctx_b.as<int16_t>(), sg.ptr<long long>(bo), sg.ptr<long long>(co), n)))
    return rc;
  std::vector<int> slots;
  if ((rc = alloc_slots(ctx, n, slots))) return rc;
  const int n_cols = ctx->main_net.plan.cond.n_cols;
  for (int i = 0; i < n; ++i)
    CK(cudaMemcpyAsync(S.pool.as<float>() + slots[i] * S.slot_stride + kSlotCond, S.cb.cond.as<float>() + (size_t)i * n_cols,
                       (size_t)n_cols * 4, cudaMemcpyDeviceToDevice, st));
  if ((rc = finish(ctx, cudaStreamSynchronize(st)))) return rc;
  for (int i = 0; i < n; ++i) {
    StreamRec r;
    r.slot = slots[i];
    r.peak = peak[i];
    ids[i] = S.next_id++;
    S.rec.emplace(ids[i], std::move(r));
  }
  return NHANS_OK;
}

int nhans_stream_step(nhans_ctx* ctx, int n, const int* ids, const int16_t* pcm, const int64_t* offs, const int* final,
                      int16_t* out_i16, float* out_f32, int64_t* out_offs) {
  return stream_step(ctx, n, ids, pcm, offs, final, out_i16, out_f32, out_offs, nullptr);
}

int nhans_stream_step_post(nhans_ctx* ctx, int n, const int* ids, const int16_t* pcm, const int64_t* offs, const int* final,
                           const float* compensate, int16_t* out_i16, float* out_f32, float* mixed_f32, float* removed_f32,
                           float* compensated_f32, int64_t* out_offs, float* snr_est) {
  PostOut post{compensate, mixed_f32, removed_f32, compensated_f32, snr_est};
  return stream_step(ctx, n, ids, pcm, offs, final, out_i16, out_f32, out_offs, &post);
}

int nhans_stream_close(nhans_ctx* ctx, int n, const int* ids) {
  if (!ctx || n < 0 || (n > 0 && !ids)) return fail(ctx, NHANS_ERR_ARG, "bad arguments");
  int rc;
  if ((rc = check_stream_ids(ctx, n, ids, false))) return rc;
  Streams& S = ctx->streams;
  for (int i = 0; i < n; ++i) {
    S.free_slots.push_back(S.rec.at(ids[i]).slot);
    S.rec.erase(ids[i]);
  }
  return NHANS_OK;
}

}  // extern "C"
