// TEST INFRASTRUCTURE ONLY - CPU interpreter of the device layer plan (nhans_b200/csrc/plan.h).
//
// It executes exactly the data structures the CUDA engine executes (padded pixel grids, k-block row
// offsets, packed fp16 weights, folded epilogue tables) with plain loops, storing activations rounded to
// fp16 like the GPU does.  tests/ use it two ways: against oracle/nhans_oracle.py it proves that plan.cc
// (geometry, folding, packing) restates N_HANS___Selective_Noise/main.py:98-242 correctly without a GPU;
// against the CUDA engine it isolates kernel bugs from plan bugs.  Never linked into libnhans_b200.so.
#include <cmath>
#include <cstdint>
#include <cstring>
#include <stdexcept>
#include <string>
#include <vector>

#include "../nhans_b200/csrc/plan.h"

using namespace nhans;

namespace {

thread_local std::string g_err;
constexpr int kMaxN = 512;               // widest layer (resblock4, the tower's last stage)

float round_f16(float v) { return f16_bits_to_f32(f32_to_f16_bits(v)); }

struct Net {
  NetPlan plan;
  std::vector<std::vector<float>> bufs;
  std::vector<std::vector<float>> wt;       // per gemm layer: [K][N] float
};

struct Units {
  std::vector<int> frame, lo, hi, utt;
};

struct Exec {
  Net main_net, tower;
  std::string json;
};

// Unpacks the weights; the activation grids are allocated by the first whole-network run (the layer-local entry points
// take their inputs from the caller).
void realise(Net& net) {
  if (net.plan.first.N > kMaxN) throw std::runtime_error("first layer wider than kMaxN");
  for (const GemmLayer& L : net.plan.gemm)
    if (L.N > kMaxN) throw std::runtime_error("layer " + L.name + " wider than kMaxN");
  net.wt.resize(net.plan.gemm.size());
  for (size_t i = 0; i < net.wt.size(); ++i) {
    const GemmLayer& L = net.plan.gemm[i];
    net.wt[i].resize((size_t)L.K * L.N);
    for (int n = 0; n < L.N; ++n)
      for (int k = 0; k < L.K; ++k) net.wt[i][(size_t)k * L.N + n] = f16_bits_to_f32(L.w[(size_t)n * L.K + k]);
  }
}

// Epilogue of one output pixel (gemm_tc.cu epilogue warps / direct_conv64_kernel tail): v[n] = the value the engine
// rounds to fp16 when it stores it, or for the head the fp32 den row.  T = float restates the engine's arithmetic for
// run_net; T = double is the layer-local reference, which also returns mag[n] = acc_abs[n] (scaled like acc) plus the
// magnitude of every epilogue term, the scale of the rounding error an fp32 evaluation of the same sum can make.
// `res` is the residual row (the same row index as the output) or null; cond_abs may be null when mag is.
template <class T>
void epilogue(const NetPlan& P, const Epilogue& E, const Units& u, const float* raw, const T* cond, const T* cond_abs, int N,
              int Wo, int unit, int ho, int wo, const float* res, const T* acc, const T* acc_abs, T* v, T* mag) {
  const size_t utt = u.utt[unit];
  const T* cb = E.cond_off >= 0 ? cond + utt * P.cond.n_cols + E.cond_off : nullptr;
  const T* cba = E.cond_off >= 0 && mag ? cond_abs + utt * P.cond.n_cols + E.cond_off : nullptr;
  const float* tf = E.tftab.empty() ? nullptr : &E.tftab[((size_t)ho * Wo + wo) * N];
  const uint16_t* t16 = E.ttab16.empty() ? nullptr : &E.ttab16[(size_t)ho * N];
  const uint16_t* f16 = E.ftab16.empty() ? nullptr : &E.ftab16[(size_t)wo * N];
  float rawv = 0.f;
  if (!E.r1_vec.empty()) {
    int frame = u.frame[unit] + ho * E.r1_sh + E.raw_oh;
    if (frame >= u.lo[unit] && frame < u.hi[unit]) rawv = raw[(size_t)frame * kBins + wo * E.r1_sw];
  }
  const float* centre = E.head ? raw + (size_t)u.frame[unit] * kBins : nullptr;
  for (int n = 0; n < N; ++n) {
    const T b = cb ? cb[n] : (T)E.bias[n];
    T x = acc[n] + b;
    if (tf) x += (T)tf[n];
    if (E.head) x = acc[n] * (T)E.res_scale[n] + b;      // inverse of the per-column weight scale (plan.cc last_dense)
    if (res) x = std::fma((T)E.res_scale[n], (T)res[n], x);
    if (!E.r1_vec.empty()) x = std::fma((T)E.r1_vec[n], (T)rawv, x);
    if (E.relu) x = x > (T)0 ? x : (T)0;
    if (centre) x = n < kBins ? x + (T)centre[n] : (T)0;
    v[n] = x;
    if (mag) {
      T m = E.head ? acc_abs[n] * std::fabs((T)E.res_scale[n]) : acc_abs[n];
      m += cba ? cba[n] : std::fabs(b);
      // the engine adds the combined table or the two fp16 tables (the row-per-thread flavours): count both
      if (tf) m += std::fabs((T)tf[n]);
      if (t16) m += std::fabs((T)f16_bits_to_f32(t16[n])) + std::fabs((T)f16_bits_to_f32(f16[n]));
      if (res) m += std::fabs((T)E.res_scale[n] * (T)res[n]);
      if (!E.r1_vec.empty()) m += std::fabs((T)E.r1_vec[n] * (T)rawv);
      if (centre && n < kBins) m += std::fabs((T)centre[n]);
      mag[n] = m;
    }
  }
}

// Stores one pixel's epilogue values like the engine: fp16 into the output grid, or the fp32 den row for the head.
void store(Net& net, const Epilogue& E, const Grid& out, int N, int unit, int ho, int wo, const float* v, float* out_f32) {
  if (E.head) {
    for (int n = 0; n < kBins; ++n) out_f32[(size_t)unit * kBins + n] = v[n];
  } else {
    float* o = &net.bufs[out.buf][(size_t)grid_pixel(out, unit, ho, wo) * out.C];
    for (int n = 0; n < N; ++n) o[n] = round_f16(v[n]);
  }
}

// Sum over the input window of the Cin = 1 convolution at one output pixel (T = float: the engine's fmaf chain).
template <class T>
void direct_acc(const DirectLayer& D, const Units& units, const float* raw, int unit, int ho, int wo, T* acc, T* acc_abs) {
  for (int n = 0; n < D.N; ++n) acc[n] = 0;
  if (acc_abs)
    for (int n = 0; n < D.N; ++n) acc_abs[n] = 0;
  for (int i = 0; i < D.kh; ++i) {
    const int r = ho * D.sh + i - D.pt;
    const int frame = units.frame[unit] + D.raw_oh + r;
    if (r < 0 || r >= D.Hin || frame < units.lo[unit] || frame >= units.hi[unit]) continue;
    for (int j = 0; j < D.kw; ++j) {
      const int f = wo * D.sw + j - D.pl;
      if (f < 0 || f >= D.Win) continue;
      const float x = raw[(size_t)frame * kBins + f];
      const float* w = &D.w[(size_t)(i * D.kw + j) * D.N];
      for (int n = 0; n < D.N; ++n) acc[n] = std::fma((T)x, (T)w[n], acc[n]);
      if (acc_abs)
        for (int n = 0; n < D.N; ++n) acc_abs[n] += std::fabs((T)x * (T)w[n]);
    }
  }
}

void run_net(Net& net, int units_n, const Units& units, const float* raw, const float* cond, float* out_f32) {
  const NetPlan& P = net.plan;
  if (net.bufs.empty()) {
    net.bufs.resize(P.bufs.size());
    for (size_t i = 0; i < net.bufs.size(); ++i) net.bufs[i].assign((size_t)P.bufs[i].pixels * P.bufs[i].C, 0.f);
  }
  {
    const DirectLayer& D = P.first;
#pragma omp parallel for schedule(dynamic, 64)
    for (long long idx = 0; idx < (long long)units_n * D.Ho * D.Wo; ++idx) {
      const int unit = (int)(idx / (D.Ho * D.Wo));
      const int rem = (int)(idx % (D.Ho * D.Wo));
      const int ho = rem / D.Wo, wo = rem % D.Wo;
      float acc[kMaxN], v[kMaxN];
      direct_acc<float>(D, units, raw, unit, ho, wo, acc, nullptr);
      epilogue<float>(P, D.epi, units, raw, cond, nullptr, D.N, D.Wo, unit, ho, wo, nullptr, acc, nullptr, v, nullptr);
      store(net, D.epi, D.out, D.N, unit, ho, wo, v, out_f32);
    }
  }
  for (size_t li = 0; li < P.gemm.size(); ++li) {
    const GemmLayer& L = P.gemm[li];
    const std::vector<float>& wt = net.wt[li];
    // compute space (plan.h): m = (ho * capacity + unit) * Wq + wo, only real output rows ho < Ho are enumerated
    const long long pitch = (long long)P.capacity * L.Wq;
    const long long per_plane = (long long)units_n * L.Wq;
    long long rows[2] = {0, 0};
    for (int a = 0; a < 2; ++a)
      if (L.a_buf[a] >= 0) rows[a] = (long long)P.bufs[L.a_buf[a]].pixels * P.bufs[L.a_buf[a]].C / L.a_rowlen[a];
#pragma omp parallel for schedule(dynamic, 32)
    for (long long idx = 0; idx < (long long)L.Ho * per_plane; ++idx) {
      const int ho = (int)(idx / per_plane);
      const long long rem = idx - (long long)ho * per_plane;
      const int unit = (int)(rem / L.Wq);
      const int wo = (int)(rem - (long long)unit * L.Wq);
      const long long m = (long long)ho * pitch + rem;
      if (wo >= L.Wo) continue;
      float acc[kMaxN] = {0}, v[kMaxN];
      for (const KGroup& g : L.groups) {
        for (int t = 0; t < g.ntaps; ++t) {
          const long long row = m + g.row_off + g.shift[t];
          if (row < 0 || row >= rows[g.map]) continue;          // TMA out-of-bounds rows read as zero
          const float* a = &net.bufs[L.a_buf[g.map]][(size_t)row * L.a_rowlen[g.map] + g.col];
          for (int kk = 0; kk < kTileK; ++kk) {
            const float av = a[kk];
            if (av == 0.f) continue;
            const float* w = &wt[(size_t)(g.bk[t] * kTileK + kk) * L.N];
            for (int n = 0; n < L.N; ++n) acc[n] += av * w[n];
          }
        }
      }
      const float* res = L.epi.res_buf >= 0 ? &net.bufs[L.epi.res_buf][(size_t)m * P.bufs[L.epi.res_buf].C] : nullptr;
      epilogue<float>(P, L.epi, units, raw, cond, nullptr, L.N, L.Wo, unit, ho, wo, res, acc, nullptr, v, nullptr);
      store(net, L.epi, L.out, L.N, unit, ho, wo, v, out_f32);
    }
  }
}

Units unit_table(const int* frame, const int* lo, const int* hi, const int* utt, int n) {
  Units u;
  u.frame.assign(frame, frame + n);
  u.lo.assign(lo, lo + n);
  u.hi.assign(hi, hi + n);
  u.utt.assign(utt, utt + n);
  return u;
}

}  // namespace

extern "C" {

const char* planexec_error() { return g_err.c_str(); }

void* planexec_create(const char* const* names, const int64_t* sizes, const float* const* data, int n, int variant,
                      int win_cap, int row_cap) {
  try {
    WeightMap w;
    for (int i = 0; i < n; ++i) w[names[i]] = std::vector<float>(data[i], data[i] + sizes[i]);
    Exec* e = new Exec;
    e->main_net.plan = build_main_plan(w, variant, win_cap);
    e->tower.plan = build_tower_plan(w, row_cap);
    realise(e->main_net);
    realise(e->tower);
    return e;
  } catch (const std::exception& ex) {
    g_err = ex.what();
    return nullptr;
  }
}

void planexec_destroy(void* h) { delete static_cast<Exec*>(h); }

const char* planexec_plan_json(void* h, int net) {
  Exec* e = static_cast<Exec*>(h);
  e->json = plan_to_json(net == 0 ? e->main_net.plan : e->tower.plan);
  return e->json.c_str();
}

int planexec_embed(void* h, const float* ctx_logmag, int R, float* emb) {
  Exec* e = static_cast<Exec*>(h);
  Net& net = e->tower;
  const int cap = net.plan.capacity;
  for (int r0 = 0; r0 < R; r0 += cap) {
    const int n = std::min(cap, R - r0);
    Units u;
    for (int i = 0; i < n; ++i) {
      u.frame.push_back((r0 + i) * kCtxFrames);
      u.lo.push_back((r0 + i) * kCtxFrames);
      u.hi.push_back((r0 + i + 1) * kCtxFrames);
      u.utt.push_back(0);
    }
    run_net(net, n, u, ctx_logmag, nullptr, nullptr);
    const Grid& g = net.plan.bufs[net.plan.pool_buf];
    for (int i = 0; i < n; ++i)
      for (int c = 0; c < 512; ++c) {
        float s = 0.f;
        for (int p = 0; p < net.plan.pool_pixels; ++p) s += net.bufs[g.buf][((size_t)i * net.plan.pool_pixels + p) * 512 + c];
        emb[(size_t)(r0 + i) * 512 + c] = s / (float)net.plan.pool_pixels;
      }
  }
  return 0;
}

int planexec_masknet(void* h, const float* logmag, const int64_t* frame_offs, int U, const float* emb_a, const float* emb_b,
                     float* denoised) {
  Exec* e = static_cast<Exec*>(h);
  Net& net = e->main_net;
  const CondTable& T = net.plan.cond;
  std::vector<float> cond((size_t)U * T.n_cols);
  for (int u = 0; u < U; ++u)
    for (int j = 0; j < T.n_cols; ++j) {
      float acc = 0.f;
      for (int k = 0; k < kEmb; ++k)
        acc = fmaf(emb_a[(size_t)u * kEmb + k], T.Pa[(size_t)k * T.n_cols + j], fmaf(emb_b[(size_t)u * kEmb + k], T.Pb[(size_t)k * T.n_cols + j], acc));
      cond[(size_t)u * T.n_cols + j] = acc + T.c[j];
    }
  const long long total = frame_offs[U];
  const int cap = net.plan.capacity;
  for (long long w0 = 0; w0 < total; w0 += cap) {
    const int n = (int)std::min<long long>(cap, total - w0);
    Units un;
    for (int i = 0; i < n; ++i) {
      const long long g = w0 + i;
      int a = 0;
      while (!(frame_offs[a] <= g && g < frame_offs[a + 1])) ++a;
      un.frame.push_back((int)g);
      un.lo.push_back((int)frame_offs[a]);
      un.hi.push_back((int)frame_offs[a + 1]);
      un.utt.push_back(a);
    }
    run_net(net, n, un, logmag, cond.data(), denoised + (size_t)w0 * kBins);
  }
  return 0;
}

// Conditioning table [U][n_cols] of the main network in double, and the sum of the magnitudes of its terms.
int planexec_cond(void* h, const float* emb_a, const float* emb_b, int U, double* cond, double* cond_abs) {
  const CondTable& T = static_cast<Exec*>(h)->main_net.plan.cond;
  for (int u = 0; u < U; ++u)
    for (int j = 0; j < T.n_cols; ++j) {
      double acc = T.c[j], mag = std::fabs((double)T.c[j]);
      for (int k = 0; k < kEmb; ++k) {
        const double pa = (double)emb_a[(size_t)u * kEmb + k] * T.Pa[(size_t)k * T.n_cols + j];
        const double pb = (double)emb_b[(size_t)u * kEmb + k] * T.Pb[(size_t)k * T.n_cols + j];
        acc += pa + pb;
        mag += std::fabs(pa) + std::fabs(pb);
      }
      cond[(size_t)u * T.n_cols + j] = acc;
      cond_abs[(size_t)u * T.n_cols + j] = mag;
    }
  return 0;
}

// The first (Cin = 1) convolution of network `net` for the n units of the given unit table, in double:
// val / S [n][Ho][Wo][N] = output before the fp16 store, and the magnitude sum bounding its rounding error.
int planexec_first(void* h, int net, const int* frame, const int* lo, const int* hi, const int* utt, int n, const float* raw,
                   const double* cond, const double* cond_abs, double* val, double* S) {
  Exec* e = static_cast<Exec*>(h);
  const NetPlan& P = (net == 0 ? e->main_net : e->tower).plan;
  const DirectLayer& D = P.first;
  const Units u = unit_table(frame, lo, hi, utt, n);
#pragma omp parallel for schedule(dynamic, 64)
  for (long long idx = 0; idx < (long long)n * D.Ho * D.Wo; ++idx) {
    const int unit = (int)(idx / (D.Ho * D.Wo));
    const int rem = (int)(idx % (D.Ho * D.Wo));
    const int ho = rem / D.Wo, wo = rem % D.Wo;
    double acc[kMaxN], acc_abs[kMaxN];
    direct_acc<double>(D, u, raw, unit, ho, wo, acc, acc_abs);
    epilogue<double>(P, D.epi, u, raw, cond, cond_abs, D.N, D.Wo, unit, ho, wo, nullptr, acc, acc_abs, val + (size_t)idx * D.N,
                     S + (size_t)idx * D.N);
  }
  return 0;
}

// One GemmLayer of network `net`, layer-local, for the n <= capacity units of the given unit table.  bufs[b] is buffer b
// of this plan (geometry of plan_json at this object's capacity) as fp32 values, null where the layer does not read it;
// errs (may be null, or hold nulls) bounds the error of each input element.  The k-group sum is taken in double, rows
// outside the A tensor read as zero like TMA's.  Outputs [n][Ho][Wo][N] (the head: [n][1][1][N], first 201 = den):
// val = the value the engine stores before its fp16 rounding, S = sum |a w| plus the epilogue term magnitudes, and
// E = sum err |w| (zero without errs).
int planexec_layer(void* h, int net, int layer, const float* const* bufs, const float* const* errs, const int* frame,
                   const int* lo, const int* hi, const int* utt, int n, const float* raw, const double* cond,
                   const double* cond_abs, double* val, double* S, double* E) {
  Exec* e = static_cast<Exec*>(h);
  Net& nd = net == 0 ? e->main_net : e->tower;
  const NetPlan& P = nd.plan;
  if (layer < 0 || layer >= (int)P.gemm.size() || n < 0 || n > P.capacity) {
    g_err = "no such layer, or more units than the capacity";
    return -1;
  }
  const GemmLayer& L = P.gemm[layer];
  for (int a = 0; a < 2; ++a)
    if (L.a_buf[a] >= 0 && !bufs[L.a_buf[a]]) { g_err = "missing A buffer of " + L.name; return -1; }
  if (L.epi.res_buf >= 0 && !bufs[L.epi.res_buf]) { g_err = "missing residual buffer of " + L.name; return -1; }
  const std::vector<float>& wt = nd.wt[layer];
  const Units u = unit_table(frame, lo, hi, utt, n);
  const long long pitch = (long long)P.capacity * L.Wq;
  long long rows[2] = {0, 0};
  for (int a = 0; a < 2; ++a)
    if (L.a_buf[a] >= 0) rows[a] = (long long)P.bufs[L.a_buf[a]].pixels * P.bufs[L.a_buf[a]].C / L.a_rowlen[a];
#pragma omp parallel for schedule(dynamic, 8)
  for (long long idx = 0; idx < (long long)n * L.Ho * L.Wo; ++idx) {
    const int unit = (int)(idx / ((long long)L.Ho * L.Wo));
    const int rem = (int)(idx % ((long long)L.Ho * L.Wo));
    const int ho = rem / L.Wo, wo = rem % L.Wo;
    const long long m = (long long)ho * pitch + (long long)unit * L.Wq + wo;
    double acc[kMaxN] = {0}, acc_abs[kMaxN] = {0}, err[kMaxN] = {0};
    for (const KGroup& g : L.groups) {
      const float* A = bufs[L.a_buf[g.map]];
      const float* Ae = errs ? errs[L.a_buf[g.map]] : nullptr;
      for (int t = 0; t < g.ntaps; ++t) {
        const long long row = m + g.row_off + g.shift[t];
        if (row < 0 || row >= rows[g.map]) continue;
        const size_t off = (size_t)row * L.a_rowlen[g.map] + g.col;
        for (int kk = 0; kk < kTileK; ++kk) {
          const double av = A[off + kk];
          const double ae = Ae ? Ae[off + kk] : 0.0;
          if (av == 0.0 && ae == 0.0) continue;
          const float* w = &wt[(size_t)(g.bk[t] * kTileK + kk) * L.N];
          const double aa = std::fabs(av);
          for (int c = 0; c < L.N; ++c) {
            acc[c] += av * w[c];
            acc_abs[c] += aa * std::fabs(w[c]);
          }
          if (ae != 0.0)
            for (int c = 0; c < L.N; ++c) err[c] += ae * std::fabs(w[c]);
        }
      }
    }
    const float* res = L.epi.res_buf >= 0 ? bufs[L.epi.res_buf] + (size_t)m * P.bufs[L.epi.res_buf].C : nullptr;
    const size_t o = (size_t)idx * L.N;
    epilogue<double>(P, L.epi, u, raw, cond, cond_abs, L.N, L.Wo, unit, ho, wo, res, acc, acc_abs, val + o, S + o);
    for (int c = 0; c < L.N; ++c) E[o + c] = err[c];
  }
  return 0;
}

int planexec_read_buffer(void* h, int net, int buf, float* out, int64_t n) {
  Exec* e = static_cast<Exec*>(h);
  Net& nd = net == 0 ? e->main_net : e->tower;
  if (buf < 0 || buf >= (int)nd.bufs.size() || n > (int64_t)nd.bufs[buf].size()) return -1;
  std::memcpy(out, nd.bufs[buf].data(), (size_t)n * sizeof(float));
  return 0;
}

}  // extern "C"
