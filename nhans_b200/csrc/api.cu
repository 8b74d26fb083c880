// Engine + C ABI (include/nhans_b200.h): one context per GPU owning a stream, the pre-packed network
// (plan.h) and the batch workspace; runs the STFT -> towers -> conditioned residual stack -> iSTFT path
// of N_HANS___Selective_Noise/apply.py:339-457 for whole batches of utterances with no host round trips
// between the stages.
#include "../../include/nhans_b200.h"

#include <algorithm>
#include <array>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <string>
#include <type_traits>
#include <vector>

#include "kernels.h"
#include "plan.h"

using namespace nhans;

namespace {

thread_local std::string g_create_error;

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

struct DBuf {
  void* p = nullptr;
  size_t cap = 0;
  cudaError_t ensure(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    size_t want = bytes + bytes / 8 + 256;
    cudaError_t e = cudaMalloc(&p, want);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
  template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

struct GemmLayerDev {
  __half* w = nullptr;
  KGroupDev* groups = nullptr;
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
  float *first_w = nullptr, *first_bias = nullptr, *first_tftab = nullptr;
  uint16_t *first_ttab16 = nullptr, *first_ftab16 = nullptr;
  float *Pa = nullptr, *Pb = nullptr, *c = nullptr;
  int *u_frame = nullptr, *u_lo = nullptr, *u_hi = nullptr, *u_utt = nullptr;
  float* convC = nullptr;           // main net: per-frame first-convolution table (kernels.h FrameConvDev)
  float* head_scratch = nullptr;    // main net: split-K partial sums of last_dense [kHeadSplit][capacity][208]
  long long crow_cap = 0;
  std::vector<void*> allocs;
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
  DBuf mix, a, b, d_mix_offs, d_a_offs, d_b_offs, d_frame_offs, d_out_offs, d_ctx_frame_offs;
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

struct Batch {
  Geometry geo;
  bool has_a = false;
  bool staged = false, done = false;
  IoSlot io[2];
  int cur = 0;                      // set the staged / running batch uses
  DBuf peak_mix, peak_a, peak_b;
  DBuf logmag, phase, den, ctxlm_a, ctxlm_b, emb_a, emb_b, cond, mixproc, removed, comp, sums, snr;
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
  DBuf tmp[8];
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

template <class T>
int upload(nhans_ctx* ctx, NetDev& net, const std::vector<T>& h, T** out) {
  *out = nullptr;
  if (h.empty()) return 0;
  void* p = nullptr;
  CK(cudaMalloc(&p, h.size() * sizeof(T)));
  net.allocs.push_back(p);
  CK(cudaMemcpyAsync(p, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
  *out = reinterpret_cast<T*>(p);
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

void free_net(NetDev& net) {
  for (void* p : net.allocs) cudaFree(p);
  net.allocs.clear();
  net.bufs.clear();
  net.layers.clear();
  net.ready = false;
}

// Allocates the activation grids (zeroed once: padding positions are never written afterwards), uploads
// packed weights and epilogue tables, encodes the TMA descriptors.
int realise_net(nhans_ctx* ctx, NetDev& net) {
  const NetPlan& P = net.plan;
  net.bufs.assign(P.bufs.size(), nullptr);
  for (size_t i = 0; i < P.bufs.size(); ++i) {
    const Grid& g = P.bufs[i];
    size_t bytes = (size_t)g.pixels * g.C * sizeof(__half);
    void* p = nullptr;
    CK(cudaMalloc(&p, bytes));
    net.allocs.push_back(p);
    CK(cudaMemsetAsync(p, 0, bytes, ctx->stream));
    net.bufs[i] = reinterpret_cast<__half*>(p);
  }
  int rc;
  if (P.cond.n_cols > 0) {
    // main net: room for the frames of one pass plus 34 virtual frames per utterance (utterances of >= 17 frames on
    // average; a pass of shorter ones falls back to the per-window kernel)
    net.crow_cap = 3LL * P.capacity + 64;
    void* p = nullptr;
    CK(cudaMalloc(&p, (size_t)4 * net.crow_cap * kBins * 64 * sizeof(float)));
    net.allocs.push_back(p);
    net.convC = reinterpret_cast<float*>(p);
  }
  if (P.cond.n_cols > 0 && !P.gemm.empty() && P.gemm.back().epi.head && !getenv("NHANS_NO_SPLITK")) {
    void* p = nullptr;
    CK(cudaMalloc(&p, (size_t)kHeadSplit * P.capacity * P.gemm.back().N * sizeof(float)));
    net.allocs.push_back(p);
    net.head_scratch = reinterpret_cast<float*>(p);
  }
  if ((rc = upload(ctx, net, P.first.w, &net.first_w))) return rc;
  if ((rc = upload(ctx, net, P.first.epi.bias, &net.first_bias))) return rc;
  if ((rc = upload(ctx, net, P.first.epi.tftab, &net.first_tftab))) return rc;
  if ((rc = upload(ctx, net, P.first.epi.ttab16, &net.first_ttab16))) return rc;
  if ((rc = upload(ctx, net, P.first.epi.ftab16, &net.first_ftab16))) return rc;
  if ((rc = upload(ctx, net, P.cond.Pa, &net.Pa))) return rc;
  if ((rc = upload(ctx, net, P.cond.Pb, &net.Pb))) return rc;
  if ((rc = upload(ctx, net, P.cond.c, &net.c))) return rc;
  net.layers.resize(P.gemm.size());
  for (size_t i = 0; i < P.gemm.size(); ++i) {
    const GemmLayer& L = P.gemm[i];
    GemmLayerDev& D = net.layers[i];
    {
      void* p = nullptr;
      CK(cudaMalloc(&p, L.w.size() * 2));
      net.allocs.push_back(p);
      CK(cudaMemcpyAsync(p, L.w.data(), L.w.size() * 2, cudaMemcpyHostToDevice, ctx->stream));
      D.w = reinterpret_cast<__half*>(p);
    }
    std::vector<KGroupDev> groups(L.groups.size());
    for (size_t j = 0; j < groups.size(); ++j) {
      const KGroup& g = L.groups[j];
      KGroupDev d;
      d.row_off = g.row_off; d.map = g.map; d.col = g.col; d.ntaps = g.ntaps; d.pad_ = 0;
      for (int t = 0; t < 4; ++t) { d.shift[t] = g.shift[t]; d.bk[t] = g.bk[t]; }
      groups[j] = d;
    }
    if ((rc = upload(ctx, net, groups, &D.groups))) return rc;
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
      if ((rc = make_map(ctx, a == 0 ? &D.mapA0 : &D.mapA1, net.bufs[buf], rowlen, elems / rowlen, 136))) return rc;
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
      uint16_t* dw = nullptr;
      if ((rc = upload(ctx, net, ww, &dw))) return rc;
      CK(cudaStreamSynchronize(ctx->stream));          // `ww` is a temporary
      D.w_walk = reinterpret_cast<__half*>(dw);
      if ((rc = make_map(ctx, &D.mapBwalk, D.w_walk, 256, 256, 256))) return rc;
    }
  }
  const int cap = P.capacity;
  for (int** p : {&net.u_frame, &net.u_lo, &net.u_hi, &net.u_utt}) {
    void* q = nullptr;
    CK(cudaMalloc(&q, sizeof(int) * (size_t)cap));
    net.allocs.push_back(q);
    *p = reinterpret_cast<int*>(q);
  }
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
    c->launches += 1;
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

struct PassInfo {                   // which frames / utterances a pass of the mask network touches
  long long w0;                     // first window (= global frame index of its centre)
  int u_first, u_last;
  const long long* d_frame_offs;
  int U;
};

// Runs `units` windows / context rows whose unit tables are already filled.
int run_net(nhans_ctx* ctx, NetDev& net, int units, const float* raw, const float* cond_table, float* out_f32,
            const PassInfo* pass = nullptr) {
  const NetPlan& P = net.plan;
  UnitTable ut{net.u_frame, net.u_lo, net.u_hi, net.u_utt};
  bool gen_first = false;
  long long gen_crow0 = 0;
  {
    const DirectLayer& D = P.first;
    DirectDev d;
    memset(&d, 0, sizeof d);
    d.units = units;
    d.kh = D.kh; d.kw = D.kw; d.sh = D.sh; d.sw = D.sw; d.pt = D.pt; d.pl = D.pl;
    d.Hin = D.Hin; d.Win = D.Win; d.raw_oh = D.raw_oh; d.Ho = D.Ho; d.Wo = D.Wo; d.N = D.N;
    d.w = net.first_w;
    d.units_tab = ut;
    d.epi = make_epi(net, D.epi, D.out, net.first_bias, net.first_tftab, nullptr, nullptr, raw, cond_table, nullptr);
    d.epi.ttab16 = reinterpret_cast<const __half*>(net.first_ttab16);
    d.epi.ftab16 = reinterpret_cast<const __half*>(net.first_ftab16);
    d.epi.tab_H = D.Ho; d.epi.tab_W = D.Wo;
    ProfScope ps(ctx, 3, 2.0 * D.macs_per_unit * units, 0);
    bool done = false;
    if (pass && net.convC && D.kh == 4 && D.kw == 4 && D.sh == 1 && D.sw == 1 && D.pt == 1 && D.pl == 1 && D.Hin == kWinFrames &&
        D.Ho == kWinFrames && D.raw_oh == -(kWinFrames / 2) && D.N == 64) {
      FrameConvDev f;
      memset(&f, 0, sizeof f);
      f.raw = raw; f.frame_offs = pass->d_frame_offs;
      f.u_first = pass->u_first; f.u_last = pass->u_last;
      f.crow0 = pass->w0 + 34LL * pass->u_first;
      const long long last = pass->w0 + units - 1 + 34LL * pass->u_last + (kWinFrames - 1);
      f.rows = (int)(last - f.crow0 + 1);
      f.crow_cap = net.crow_cap;
      f.w = net.first_w;
      f.bias = d.epi.bias; f.bias_stride = d.epi.bias_stride; f.ftab16 = d.epi.ftab16;
      f.C = net.convC;
      if (f.rows <= net.crow_cap) {
        // (expanding the pass in slices so that a slice's table stays L2-resident was measured: no gain)
        CK(launch_frame_conv(ctx->stream, f));
        // the row-walk kernel of the next layer builds its A operand from the table (conv_walk.cu kWalkGen); otherwise
        // the table is expanded into the (window, row) activation tensor here
        gen_first = ctx->use_walk && ctx->use_gen && !P.gemm.empty() && P.gemm[0].walk && net.layers[0].w_walk &&
                    P.gemm[0].a_buf[0] == D.out.buf && D.epi.relu && d.epi.ttab16;
        if (gen_first) {
          gen_crow0 = f.crow0;
        } else {
          CK(launch_window_expand(ctx->stream, d, net.convC, f.crow0, net.crow_cap, 0, units));
          ctx->launches += 1;
        }
        done = true;
      }
    }
    if (!done) CK(launch_direct_conv(ctx->stream, d));
  }
  for (size_t i = 0; i < P.gemm.size(); ++i) {
    const GemmLayer& L = P.gemm[i];
    const GemmLayerDev& D = net.layers[i];
    GemmDev g;
    memset(&g, 0, sizeof g);
    long long M = (long long)units * L.Ho * L.Wq;
    if ((long long)P.capacity * L.Ho * L.Wq > 0x7fffffffLL) return fail(ctx, NHANS_ERR_ARG, "too many rows in one pass");
    g.M = (int)M; g.plane_pitch = P.capacity * L.Wq; g.plane_rows = units * L.Wq; g.N = L.N; g.BN = L.BN; g.num_kb = (int)L.kb.size(); g.num_groups = (int)L.groups.size(); g.groups = D.groups;
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
        wd.gen_C = net.convC; wd.gen_crow0 = gen_crow0; wd.gen_crow_cap = net.crow_cap;
        wd.gen_ttab16 = reinterpret_cast<const __half*>(net.first_ttab16);
      }
      cudaError_t le = launch_walk(ctx->stream, ctx->n_sm, D.mapA0, D.mapBwalk, wd);
      if (le != cudaSuccess)
        return fail(ctx, NHANS_ERR_CUDA, "launch of row-walk layer " + L.name + ": " + cudaGetErrorString(le));
      continue;
    }
    {
      cudaError_t le = launch_gemm(ctx->stream, ctx->n_sm, D.mapA0, D.mapA1, D.mapB, D.mapBhalf, g);
      if (le != cudaSuccess)
        return fail(ctx, NHANS_ERR_CUDA, "launch of layer " + L.name + " (M " + std::to_string(g.M) + ", BN " + std::to_string(g.BN) + "): " + cudaGetErrorString(le));
      if (split_head) {
        CK(launch_head_reduce(ctx->stream, net.head_scratch, kHeadSplit, units, L.N, D.res_scale, D.bias, raw, net.u_frame, out_f32));
        ctx->launches += 1;
      }
    }
  }
  return 0;
}

// Embedding tower over R context rows of ctx_logmag (device, [R][200][201]) -> emb (device, [R][512]).
int run_tower(nhans_ctx* ctx, const float* ctx_logmag, int R, float* emb) {
  NetDev& net = ctx->tower;
  const int cap = net.plan.capacity;
  for (int r0 = 0; r0 < R; r0 += cap) {
    const int n = std::min(cap, R - r0);
    CK(launch_units_rows(ctx->stream, r0, n, kCtxFrames, net.u_frame, net.u_lo, net.u_hi, net.u_utt));
    ctx->launches += 1;
    int rc = run_net(ctx, net, n, ctx_logmag, nullptr, nullptr);
    if (rc) return rc;
    ProfScope ps(ctx, 4, 0, 0);
    CK(launch_mean_pool(ctx->stream, net.bufs[net.plan.pool_buf], n, net.plan.pool_pixels, 512, emb + (size_t)r0 * 512));
  }
  return 0;
}

// Mask network over all frames (device logmag rows) -> denoised rows.
int run_masknet(nhans_ctx* ctx, const float* logmag, const long long* d_frame_offs, const long long* h_frame_offs, int U,
                long long total_frames, const float* cond_table, float* den) {
  NetDev& net = ctx->main_net;
  const int cap = net.plan.capacity;
  if (total_frames > 0x7fffffffLL) return fail(ctx, NHANS_ERR_ARG, "too many frames in one batch");
  for (long long w0 = 0; w0 < total_frames; w0 += cap) {
    const int n = (int)std::min<long long>(cap, total_frames - w0);
    CK(launch_units_main(ctx->stream, d_frame_offs, U, (int)w0, n, net.u_frame, net.u_lo, net.u_hi, net.u_utt));
    ctx->launches += 1;
    PassInfo pi;
    pi.w0 = w0; pi.d_frame_offs = d_frame_offs; pi.U = U;
    // utterances of the first / last window of the pass: largest u with frame_offs[u] <= frame
    pi.u_first = (int)(std::upper_bound(h_frame_offs, h_frame_offs + U + 1, w0) - h_frame_offs) - 1;
    pi.u_last = (int)(std::upper_bound(h_frame_offs, h_frame_offs + U + 1, w0 + n - 1) - h_frame_offs) - 1;
    int rc = run_net(ctx, net, n, logmag, cond_table, den + (size_t)w0 * kBins, &pi);
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

int to_device_offs(nhans_ctx* ctx, DBuf& d, const std::vector<long long>& h, cudaStream_t stream = nullptr) {
  CK(d.ensure(h.size() * sizeof(long long)));
  CK(cudaMemcpyAsync(d.p, h.data(), h.size() * sizeof(long long), cudaMemcpyHostToDevice, stream ? stream : ctx->stream));
  return 0;
}

int need_weights(nhans_ctx* ctx) {
  if (!ctx->main_net.ready || !ctx->tower.ready) return fail(ctx, NHANS_ERR_STATE, "nhans_load_weights has not been called");
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
  auto clips = [&](DBuf& d, const T* x, const int64_t* offs, long long n) {
    CK(d.ensure(n * sizeof(T) + 32));
    CK(cudaMemcpyAsync(d.p, x + offs[0], n * sizeof(T), cudaMemcpyHostToDevice, stream));
    return 0;
  };
  const int U = g.U;
  int rc;
  if ((rc = clips(io.mix, mix, mix_offs, g.mix_offs[U]))) return rc;
  if ((rc = clips(io.b, ctx_b, b_offs, g.b_offs[U]))) return rc;
  if (ctx_a) {
    if ((rc = clips(io.a, ctx_a, a_offs, g.a_offs[U]))) return rc;
    if ((rc = to_device_offs(ctx, io.d_a_offs, g.a_offs, stream))) return rc;
  }
  if ((rc = to_device_offs(ctx, io.d_mix_offs, g.mix_offs, stream))) return rc;
  if ((rc = to_device_offs(ctx, io.d_b_offs, g.b_offs, stream))) return rc;
  if ((rc = to_device_offs(ctx, io.d_frame_offs, g.frame_offs, stream))) return rc;
  if ((rc = to_device_offs(ctx, io.d_out_offs, g.out_offs, stream))) return rc;
  if ((rc = to_device_offs(ctx, io.d_ctx_frame_offs, g.ctx_frame_offs, stream))) return rc;
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
  const size_t cbytes = (size_t)U * kCtxFrames * kBins * 4;
  const int n_cols = ctx->main_net.plan.cond.n_cols;
  cudaStream_t st = ctx->stream;
  CK(b.peak_mix.ensure(sizeof(int) * U));
  CK(b.logmag.ensure(sbytes + 4));
  CK(b.phase.ensure(2 * sbytes + 8));          // unit phasors (float2 per bin) between the two transforms
  CK(b.den.ensure(sbytes + 4));
  CK(b.ctxlm_b.ensure(cbytes));
  CK(b.emb_b.ensure((size_t)U * 512 * 4));
  CK(b.cond.ensure((size_t)U * n_cols * 4));
  if (b.has_a) {
    CK(b.ctxlm_a.ensure(cbytes));
    CK(b.emb_a.ensure((size_t)U * 512 * 4));
  }
  if (pcm) {
    CK(b.peak_a.ensure(sizeof(int) * U));
    CK(b.peak_b.ensure(sizeof(int) * U));
    CK(launch_peaks(st, io.mix.as<int16_t>(), io.d_mix_offs.as<long long>(), U, b.peak_mix.as<int>()));
    CK(launch_peaks(st, io.b.as<int16_t>(), io.d_b_offs.as<long long>(), U, b.peak_b.as<int>()));
    ctx->launches += 2;
  } else {
    CK(cudaMemsetAsync(b.peak_mix.p, 0, sizeof(int) * U, st));     // the inverse STFT reads it; no int16 output here
  }
  {
    ProfScope ps(ctx, 1, 0, (double)sizeof(T) * g.mix_offs[U] + 3.0 * sbytes);
    CK(launch_stft_of(st, io.mix.as<T>(), io.d_mix_offs.as<long long>(), io.d_frame_offs.as<long long>(), U,
                      b.peak_mix.as<int>(), g.max_frames, b.logmag.as<float>(), b.phase.as<float>(), true));
  }
  {
    ProfScope ps(ctx, 4, 0, 0);
    CK(launch_stft_of(st, io.b.as<T>(), io.d_b_offs.as<long long>(), io.d_ctx_frame_offs.as<long long>(), U,
                      b.peak_b.as<int>(), kCtxFrames, b.ctxlm_b.as<float>(), nullptr, false));
  }
  const float* emb_a = ctx->silent_emb.as<float>();
  int stride_a = 0;
  int rc;
  if (b.has_a) {
    if (pcm) {
      CK(launch_peaks(st, io.a.as<int16_t>(), io.d_a_offs.as<long long>(), U, b.peak_a.as<int>()));
      ctx->launches += 1;
    }
    {
      ProfScope ps(ctx, 4, 0, 0);
      CK(launch_stft_of(st, io.a.as<T>(), io.d_a_offs.as<long long>(), io.d_ctx_frame_offs.as<long long>(), U,
                        b.peak_a.as<int>(), kCtxFrames, b.ctxlm_a.as<float>(), nullptr, false));
    }
    // embedding towers: once per distinct context clip (SURVEY.md F6), not once per window
    if ((rc = run_tower(ctx, b.ctxlm_a.as<float>(), U, b.emb_a.as<float>()))) return rc;
    emb_a = b.emb_a.as<float>();
    stride_a = 512;
  }
  if ((rc = run_tower(ctx, b.ctxlm_b.as<float>(), U, b.emb_b.as<float>()))) return rc;
  {
    ProfScope ps(ctx, 4, 0, 0);
    CK(launch_cond_table(st, emb_a, stride_a, b.emb_b.as<float>(), 512, U, ctx->main_net.Pa, ctx->main_net.Pb,
                         ctx->main_net.c, n_cols, b.cond.as<float>()));
  }
  return run_masknet(ctx, b.logmag.as<float>(), io.d_frame_offs.as<long long>(), g.frame_offs.data(), U, g.total_frames,
                     b.cond.as<float>(), b.den.as<float>());
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
  CK(ctx->tmp[0].ensure(total * sizeof(T) + 32));
  CK(cudaMemcpyAsync(ctx->tmp[0].p, x + offs[0], total * sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
  if ((rc = to_device_offs(ctx, ctx->tmp[1], g.mix_offs))) return rc;
  if ((rc = to_device_offs(ctx, ctx->tmp[2], g.frame_offs))) return rc;
  const size_t sbytes = (size_t)g.total_frames * kBins * 4;
  CK(ctx->tmp[4].ensure(sbytes + 4));
  CK(ctx->tmp[5].ensure(sbytes + 4));
  if (pcm) {
    CK(ctx->tmp[3].ensure(sizeof(int) * U));
    CK(launch_peaks(ctx->stream, ctx->tmp[0].as<int16_t>(), ctx->tmp[1].as<long long>(), U, ctx->tmp[3].as<int>()));
  }
  {
    ProfScope ps(ctx, 1, 0, (double)sizeof(T) * total + 2.0 * sbytes);
    CK(launch_stft_of(ctx->stream, ctx->tmp[0].as<T>(), ctx->tmp[1].as<long long>(), ctx->tmp[2].as<long long>(), U,
                      ctx->tmp[3].as<int>(), g.max_frames, ctx->tmp[4].as<float>(), ctx->tmp[5].as<float>(), false));
  }
  if (logmag) CK(cudaMemcpyAsync(logmag, ctx->tmp[4].p, sbytes, cudaMemcpyDeviceToHost, ctx->stream));
  if (phase) CK(cudaMemcpyAsync(phase, ctx->tmp[5].p, sbytes, cudaMemcpyDeviceToHost, ctx->stream));
  if (peak) CK(cudaMemcpyAsync(peak, ctx->tmp[3].p, sizeof(int) * U, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
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
  cudaStreamSynchronize(ctx->stream);
  free_net(ctx->main_net);
  free_net(ctx->tower);
  Batch& b = ctx->batch;
  if (ctx->h2d_stream) cudaStreamSynchronize(ctx->h2d_stream);
  if (ctx->d2h_stream) cudaStreamSynchronize(ctx->d2h_stream);
  for (IoSlot& io : b.io) {
    for (DBuf* d : {&io.mix, &io.a, &io.b, &io.d_mix_offs, &io.d_a_offs, &io.d_b_offs, &io.d_frame_offs, &io.d_out_offs,
                    &io.d_ctx_frame_offs, &io.out_i16, &io.out_f32})
      d->release();
    for (cudaEvent_t ev : {io.uploaded, io.consumed, io.drained}) if (ev) cudaEventDestroy(ev);
  }
  for (DBuf* d : {&b.peak_mix, &b.peak_a, &b.peak_b, &b.logmag, &b.phase, &b.den, &b.ctxlm_a,
                  &b.ctxlm_b, &b.emb_a, &b.emb_b, &b.cond, &b.mixproc, &b.removed, &b.comp, &b.sums,
                  &b.snr, &ctx->silent_emb})
    d->release();
  for (auto& t : ctx->tmp) t.release();
  for (auto& ev : ctx->events) if (ev) cudaEventDestroy(ev);
  for (auto& r : ctx->prof) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
  for (auto& ev : ctx->ev_pool) cudaEventDestroy(ev);
  for (auto& ev : ctx->tl) for (auto& e : ev) if (e) cudaEventDestroy(e);
  if (ctx->tl_origin) cudaEventDestroy(ctx->tl_origin);
  if (ctx->err_flag_host) cudaFreeHost(ctx->err_flag_host);
  if (ctx->stream) cudaStreamDestroy(ctx->stream);
  if (ctx->h2d_stream) cudaStreamDestroy(ctx->h2d_stream);
  if (ctx->d2h_stream) cudaStreamDestroy(ctx->d2h_stream);
  delete ctx;
}

int nhans_load_weights(nhans_ctx* ctx, const char* const* names, const int64_t* sizes, const float* const* data, int n) {
  if (!ctx || !names || !sizes || !data || n <= 0) return fail(ctx, NHANS_ERR_ARG, "bad arguments");
  CK(cudaSetDevice(ctx->device));
  WeightMap w;
  for (int i = 0; i < n; ++i) w[names[i]] = std::vector<float>(data[i], data[i] + sizes[i]);
  free_net(ctx->main_net);
  free_net(ctx->tower);
  ctx->silent_ready = false;
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
  std::vector<long long> ho(offs, offs + U + 1), oo(U + 1, 0);
  for (int u = 0; u < U; ++u) {
    long long n = ho[u + 1] - ho[u];
    if (trim && n >= 400) n -= (n - 400) % 160;
    oo[u + 1] = oo[u] + n;
  }
  const long long total = ho[U] - ho[0];
  CK(ctx->tmp[0].ensure(total * 2 + 32));
  CK(cudaMemcpyAsync(ctx->tmp[0].p, pcm + ho[0], total * 2, cudaMemcpyHostToDevice, ctx->stream));
  std::vector<long long> rel(U + 1);
  for (int u = 0; u <= U; ++u) rel[u] = ho[u] - ho[0];
  int rc;
  if ((rc = to_device_offs(ctx, ctx->tmp[1], rel))) return rc;
  if ((rc = to_device_offs(ctx, ctx->tmp[2], oo))) return rc;
  CK(ctx->tmp[3].ensure(sizeof(int) * U));
  CK(ctx->tmp[4].ensure(oo[U] * 4 + 4));
  CK(launch_peaks(ctx->stream, ctx->tmp[0].as<int16_t>(), ctx->tmp[1].as<long long>(), U, ctx->tmp[3].as<int>()));
  CK(launch_normalise(ctx->stream, ctx->tmp[0].as<int16_t>(), ctx->tmp[1].as<long long>(), ctx->tmp[2].as<long long>(), U,
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
    CK(launch_eval_loss(ctx->stream, ctx->tmp[0].as<float>(), ctx->tmp[1].as<float>(), n_frames, ctx->tmp[2].as<float>()));
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
  cudaError_t e = cudaStreamSynchronize(ctx->stream);
  if ((rc = check_kernel_flag(ctx))) return rc;
  CK(e);
  return NHANS_OK;
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
  if ((rc = to_device_offs(ctx, ctx->tmp[5], fo))) return rc;
  CK(cudaMemcpyAsync(ctx->tmp[0].p, logmag, sbytes, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(ctx->tmp[2].p, emb_a, (size_t)U * 512 * 4, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(ctx->tmp[3].p, emb_b, (size_t)U * 512 * 4, cudaMemcpyHostToDevice, ctx->stream));
  CK(launch_cond_table(ctx->stream, ctx->tmp[2].as<float>(), 512, ctx->tmp[3].as<float>(), 512, U, ctx->main_net.Pa,
                       ctx->main_net.Pb, ctx->main_net.c, n_cols, ctx->tmp[4].as<float>()));
  if ((rc = run_masknet(ctx, ctx->tmp[0].as<float>(), ctx->tmp[5].as<long long>(), fo.data(), U, total, ctx->tmp[4].as<float>(),
                        ctx->tmp[1].as<float>())))
    return rc;
  CK(cudaMemcpyAsync(denoised, ctx->tmp[1].p, sbytes, cudaMemcpyDeviceToHost, ctx->stream));
  cudaError_t e = cudaStreamSynchronize(ctx->stream);
  if ((rc = check_kernel_flag(ctx))) return rc;
  CK(e);
  return NHANS_OK;
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
  int rc;
  if ((rc = to_device_offs(ctx, ctx->tmp[2], fo))) return rc;
  if ((rc = to_device_offs(ctx, ctx->tmp[3], oo))) return rc;
  std::vector<int> pk(U, 0);
  if (peak) for (int u = 0; u < U; ++u) pk[u] = peak[u];
  CK(ctx->tmp[4].ensure(sizeof(int) * U));
  CK(cudaMemcpyAsync(ctx->tmp[4].p, pk.data(), sizeof(int) * U, cudaMemcpyHostToDevice, ctx->stream));
  CK(ctx->tmp[5].ensure(oo[U] * 4 + 4));
  CK(ctx->tmp[6].ensure(oo[U] * 2 + 4));
  {
    ProfScope ps(ctx, 2, 0, 2.0 * sbytes + (wav_f32 ? 4.0 : 0.0) * oo[U] + (wav_i16 ? 2.0 : 0.0) * oo[U]);
    CK(launch_istft(ctx->stream, ctx->tmp[0].as<float>(), ctx->tmp[1].as<float>(), ctx->tmp[2].as<long long>(),
                    ctx->tmp[3].as<long long>(), U, ctx->tmp[4].as<int>(), max_frames, wav_f32 ? ctx->tmp[5].as<float>() : nullptr,
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
  if (ctx_a && !a_offs) return fail(ctx, NHANS_ERR_ARG, "ctx_a given without offsets");
  if (!ctx_a && ctx->variant != NHANS_VARIANT_SELECTIVE_NOISE)
    return fail(ctx, NHANS_ERR_ARG, "the separator needs both context recordings");
  CK(cudaSetDevice(ctx->device));
  int rc;
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
  {
    ProfScope ps(ctx, 2, 0, 3.0 * g.total_frames * kBins * 4 + 6.0 * g.total_out);
    CK(launch_istft(ctx->stream, b.den.as<float>(), b.phase.as<float>(), io.d_frame_offs.as<long long>(),
                    io.d_out_offs.as<long long>(), g.U, b.peak_mix.as<int>(), g.max_frames, io.out_f32.as<float>(),
                    io.out_i16.as<int16_t>(), true));
  }
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
    ProfScope ps(ctx, 2, 0, 3.0 * g.total_frames * kBins * 4 + 4.0 * g.total_out);
    CK(launch_istft(ctx->stream, b.logmag.as<float>(), b.phase.as<float>(), io.d_frame_offs.as<long long>(),
                    io.d_out_offs.as<long long>(), g.U, b.peak_mix.as<int>(), g.max_frames, b.mixproc.as<float>(), nullptr, true));
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
    CK(launch_istft_post(ctx->stream, b.den.as<float>(), b.logmag.as<float>(), b.phase.as<float>(), io.d_frame_offs.as<long long>(),
                         io.d_out_offs.as<long long>(), g.U, g.max_frames, nullptr, b.mixproc.as<float>(), b.removed.as<float>(),
                         b.sums.as<double>(), true));
  }
  {
    ProfScope ps(ctx, 4, 0, 0);
    CK(launch_compensate(ctx->stream, io.out_f32.as<float>(), b.removed.as<float>(), io.d_out_offs.as<long long>(), g.U,
                         b.sums.as<double>(), compensate, ac, compensated_f32 ? b.comp.as<float>() : nullptr, b.snr.as<float>()));
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
  if (ctx_a && !a_offs) return fail(ctx, NHANS_ERR_ARG, "ctx_a given without offsets");
  if (!ctx_a && ctx->variant != NHANS_VARIANT_SELECTIVE_NOISE) return fail(ctx, NHANS_ERR_ARG, "the separator needs both context recordings");
  CK(cudaSetDevice(ctx->device));
  int rc;
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
  const double istft_bytes = 3.0 * g.total_frames * kBins * 4 + 4.0 * g.total_out;
  CK(io.out_f32.ensure(g.total_out * 4 + 16));
  if (out_f32) {
    ProfScope ps(ctx, 2, 0, istft_bytes);
    CK(launch_istft(st, b.den.as<float>(), b.phase.as<float>(), io.d_frame_offs.as<long long>(), io.d_out_offs.as<long long>(), U,
                    b.peak_mix.as<int>(), g.max_frames, io.out_f32.as<float>(), nullptr, true));
    CK(cudaMemcpyAsync(out_f32, io.out_f32.p, g.total_out * 4, cudaMemcpyDeviceToHost, st));
  }
  if (mixproc_f32) {
    CK(b.mixproc.ensure(g.total_out * 4 + 16));
    ProfScope ps(ctx, 2, 0, istft_bytes);
    CK(launch_istft(st, b.logmag.as<float>(), b.phase.as<float>(), io.d_frame_offs.as<long long>(), io.d_out_offs.as<long long>(), U,
                    b.peak_mix.as<int>(), g.max_frames, b.mixproc.as<float>(), nullptr, true));
    CK(cudaMemcpyAsync(mixproc_f32, b.mixproc.p, g.total_out * 4, cudaMemcpyDeviceToHost, st));
  }
  cudaError_t e = cudaStreamSynchronize(st);
  if ((rc = check_kernel_flag(ctx))) return rc;
  CK(e);
  return NHANS_OK;
}

int nhans_sync(nhans_ctx* ctx) {
  if (!ctx) return NHANS_ERR_ARG;
  cudaSetDevice(ctx->device);
  cudaError_t e = cudaStreamSynchronize(ctx->stream);
  cudaError_t e1 = cudaStreamSynchronize(ctx->h2d_stream);
  cudaError_t e2 = cudaStreamSynchronize(ctx->d2h_stream);
  for (IoSlot& io : ctx->batch.io) io.d2h_pending = false;
  int rc;
  if ((rc = check_kernel_flag(ctx))) return rc;
  CK(e);
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
    int rc;
    if ((rc = check_kernel_flag(ctx))) return rc;
    CK(e);
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

}  // extern "C"
