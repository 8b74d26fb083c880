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
#include <string>
#include <vector>

#include "../nhans_b200/csrc/plan.h"

using namespace nhans;

namespace {

thread_local std::string g_err;

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

void realise(Net& net) {
  net.bufs.resize(net.plan.bufs.size());
  for (size_t i = 0; i < net.bufs.size(); ++i) net.bufs[i].assign((size_t)net.plan.bufs[i].pixels * net.plan.bufs[i].C, 0.f);
  net.wt.resize(net.plan.gemm.size());
  for (size_t i = 0; i < net.wt.size(); ++i) {
    const GemmLayer& L = net.plan.gemm[i];
    net.wt[i].resize((size_t)L.K * L.N);
    for (int n = 0; n < L.N; ++n)
      for (int k = 0; k < L.K; ++k) net.wt[i][(size_t)k * L.N + n] = f16_bits_to_f32(L.w[(size_t)n * L.K + k]);
  }
}

struct EpiCtx {
  const Net* net;
  const Units* units;
  const float* raw;
  const float* cond;      // [U][n_cols]
  float* out_f32;
};

// Shared epilogue (gemm_tc.cu epilogue warps / direct_conv64_kernel tail).
void epilogue(const EpiCtx& c, const Epilogue& E, const Grid& out, int N, int Wo, int unit, int ho, int wo, long long res_row,
              const float* acc, std::vector<std::vector<float>>& bufs) {
  const int utt = c.units->utt[unit];
  const float* bias = E.cond_off >= 0 ? c.cond + (size_t)utt * c.net->plan.cond.n_cols + E.cond_off : E.bias.data();
  float rawv = 0.f;
  if (!E.r1_vec.empty()) {
    int frame = c.units->frame[unit] + ho * E.r1_sh + E.raw_oh;
    if (frame >= c.units->lo[unit] && frame < c.units->hi[unit]) rawv = c.raw[(size_t)frame * kBins + wo * E.r1_sw];
  }
  for (int n = 0; n < N; ++n) {
    float v = acc[n] + bias[n];
    if (!E.tftab.empty()) v += E.tftab[((size_t)ho * Wo + wo) * N + n];
    if (E.head) v = acc[n] * E.res_scale[n] + bias[n];      // inverse of the per-column weight scale (plan.cc last_dense)
    if (E.res_buf >= 0) v = fmaf(E.res_scale[n], bufs[E.res_buf][(size_t)res_row * c.net->plan.bufs[E.res_buf].C + n], v);
    if (!E.r1_vec.empty()) v = fmaf(E.r1_vec[n], rawv, v);
    if (E.relu) v = v > 0.f ? v : 0.f;
    if (E.head) {
      if (n < kBins) c.out_f32[(size_t)unit * kBins + n] = v + c.raw[(size_t)c.units->frame[unit] * kBins + n];
    } else {
      bufs[out.buf][(size_t)grid_pixel(out, unit, ho, wo) * out.C + n] = round_f16(v);
    }
  }
}

void run_net(Net& net, int units_n, const Units& units, const float* raw, const float* cond, float* out_f32) {
  const NetPlan& P = net.plan;
  EpiCtx c{&net, &units, raw, cond, out_f32};
  {
    const DirectLayer& D = P.first;
#pragma omp parallel for schedule(dynamic, 64)
    for (long long idx = 0; idx < (long long)units_n * D.Ho * D.Wo; ++idx) {
      const int unit = (int)(idx / (D.Ho * D.Wo));
      const int rem = (int)(idx % (D.Ho * D.Wo));
      const int ho = rem / D.Wo, wo = rem % D.Wo;
      float acc[64] = {0};
      for (int i = 0; i < D.kh; ++i) {
        const int r = ho * D.sh + i - D.pt;
        const int frame = units.frame[unit] + D.raw_oh + r;
        if (r < 0 || r >= D.Hin || frame < units.lo[unit] || frame >= units.hi[unit]) continue;
        for (int j = 0; j < D.kw; ++j) {
          const int f = wo * D.sw + j - D.pl;
          if (f < 0 || f >= D.Win) continue;
          const float x = raw[(size_t)frame * kBins + f];
          const float* w = &D.w[(size_t)(i * D.kw + j) * D.N];
          for (int n = 0; n < D.N; ++n) acc[n] = fmaf(x, w[n], acc[n]);
        }
      }
      epilogue(c, D.epi, D.out, D.N, D.Wo, unit, ho, wo, 0, acc, net.bufs);
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
      std::vector<float> acc(L.N, 0.f);
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
      epilogue(c, L.epi, L.out, L.N, L.Wo, unit, ho, wo, m, acc.data(), net.bufs);
    }
  }
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

int planexec_read_buffer(void* h, int net, int buf, float* out, int64_t n) {
  Exec* e = static_cast<Exec*>(h);
  Net& nd = net == 0 ? e->main_net : e->tower;
  if (buf < 0 || buf >= (int)nd.bufs.size() || n > (int64_t)nd.bufs[buf].size()) return -1;
  std::memcpy(out, nd.bufs[buf].data(), (size_t)n * sizeof(float));
  return 0;
}

}  // extern "C"
