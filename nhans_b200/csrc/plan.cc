// Builds the device layer plan from TF-named weights: geometry, k-block tables, weight packing and
// the batch-norm / bias / embedding folding of SURVEY.md App. A.6.  Host-only C++.
//
// Follows N_HANS___Selective_Noise/main.py:102-124 (noise_resnet_block), :126-187 (resnet_block with
// cont_embed :127-137 and process_noise_t_f :139-159), :189-242 (towers, stack, head) and
// blocks.py:23-48 (dense / conv2d), :104-108 (eval batch-norm, eps 1e-3).
#include "plan.h"

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <stdexcept>

namespace nhans {

void same_pads(int n, int k, int s, int* out, int* before, int* after) {
  int o = (n + s - 1) / s;
  int pad = std::max((o - 1) * s + k - n, 0);
  *out = o;
  *before = pad / 2;
  *after = pad - pad / 2;
}

uint16_t f32_to_f16_bits(float f) {
  uint32_t x;
  std::memcpy(&x, &f, 4);
  uint32_t sign = (x >> 16) & 0x8000u;
  uint32_t mant = x & 0x7fffffu;
  int exp = (int)((x >> 23) & 0xff);
  if (exp == 0xff) return (uint16_t)(sign | 0x7c00u | (mant ? 0x200u : 0));
  int e = exp - 127 + 15;
  if (e >= 31) return (uint16_t)(sign | 0x7c00u);
  if (e <= 0) {
    if (e < -10) return (uint16_t)sign;
    mant |= 0x800000u;
    int shift = 14 - e;
    uint32_t half = mant >> shift;
    uint32_t rem = mant & ((1u << shift) - 1);
    uint32_t mid = 1u << (shift - 1);
    if (rem > mid || (rem == mid && (half & 1))) half++;
    return (uint16_t)(sign | half);
  }
  uint32_t half = ((uint32_t)e << 10) | (mant >> 13);
  uint32_t rem = mant & 0x1fffu;
  if (rem > 0x1000u || (rem == 0x1000u && (half & 1))) half++;
  return (uint16_t)(sign | half);
}

float f16_bits_to_f32(uint16_t h) {
  uint32_t sign = (uint32_t)(h & 0x8000u) << 16;
  uint32_t exp = (h >> 10) & 0x1f;
  uint32_t mant = h & 0x3ffu;
  uint32_t x;
  if (exp == 0) {
    if (mant == 0) {
      x = sign;
    } else {
      int e = -1;
      do { mant <<= 1; e++; } while (!(mant & 0x400u));
      x = sign | ((uint32_t)(127 - 15 - e) << 23) | ((mant & 0x3ffu) << 13);
    }
  } else if (exp == 31) {
    x = sign | 0x7f800000u | (mant << 13);
  } else {
    x = sign | ((exp - 15 + 127) << 23) | (mant << 13);
  }
  float f;
  std::memcpy(&f, &x, 4);
  return f;
}

namespace {

const std::vector<float>& get(const WeightMap& w, const std::string& name, size_t expect) {
  auto it = w.find(name);
  if (it == w.end()) throw std::runtime_error("missing variable '" + name + "'");
  if (it->second.size() != expect)
    throw std::runtime_error("variable '" + name + "' has " + std::to_string(it->second.size()) +
                             " elements, expected " + std::to_string(expect));
  return it->second;
}

struct Affine {                      // y = x * s + o  (eval batch-norm, blocks.py:104-108)
  std::vector<double> s, o;
};

Affine fold_bn(const WeightMap& w, const std::string& scope, int C) {
  const auto& beta = get(w, scope + "/beta", C);
  const auto& gamma = get(w, scope + "/gamma", C);
  const auto& mean = get(w, scope + "/pop_mean", C);
  const auto& var = get(w, scope + "/pop_variance", C);
  Affine a;
  a.s.resize(C);
  a.o.resize(C);
  for (int c = 0; c < C; ++c) {
    // tf.nn.batch_normalization: inv = rsqrt(var + eps) * gamma; y = x * inv + (beta - mean * inv)
    double inv = (double)gamma[c] / std::sqrt((double)var[c] + 0.001);
    a.s[c] = inv;
    a.o[c] = (double)beta[c] - (double)mean[c] * inv;
  }
  return a;
}

// cont_embed(n, C, scope), main.py:127-137: range(n) -> dense1 -> BN -> ReLU -> dense2 -> BN -> ReLU -> dense3
std::vector<double> cont_embed(const WeightMap& w, const std::string& scope, int n, int C) {
  const auto& w1 = get(w, scope + "_dense1/w", 50);
  const auto& w2 = get(w, scope + "_dense2/w", 2500);
  const auto& w3 = get(w, scope + "_dense3/w", (size_t)50 * C);
  Affine b1 = fold_bn(w, scope + scope + "_dense1", 50);
  Affine b2 = fold_bn(w, scope + scope + "_dense2", 50);
  std::vector<double> out((size_t)n * C);
  for (int i = 0; i < n; ++i) {
    double h1[50], h2[50];
    for (int j = 0; j < 50; ++j) h1[j] = std::max(0.0, (double)i * w1[j] * b1.s[j] + b1.o[j]);
    for (int j = 0; j < 50; ++j) {
      double a = 0;
      for (int k = 0; k < 50; ++k) a += h1[k] * w2[k * 50 + j];
      h2[j] = std::max(0.0, a * b2.s[j] + b2.o[j]);
    }
    for (int c = 0; c < C; ++c) {
      double a = 0;
      for (int k = 0; k < 50; ++k) a += h2[k] * w3[(size_t)k * C + c];
      out[(size_t)i * C + c] = a;
    }
  }
  return out;
}

struct BlockSpec {
  std::string scope;
  int kh, kw, sh, sw, C;
};

struct BlockGeom {
  int H, W, Cin;                       // input
  int Ho, Wo;                          // output
  int pt, pb, pl, pr;                  // conv1 pads
  int pt2, pb2, pl2, pr2;              // conv2 pads
  int Hq, Wq;                          // compute pitch shared by every buffer the block reads
};

int floordiv(int a, int b) { return (a >= 0) ? a / b : -((-a + b - 1) / b); }

// Row offset of the input pixel (ho * sh + dy, wo * sw + dx) relative to compute row (ho, wo).
int32_t tap_offset(const Grid& g, int dy, int dx) {
  int y0 = dy + g.oy, x0 = dx + g.ox;
  int qy = floordiv(y0, g.sh), qx = floordiv(x0, g.sw);
  int py = y0 - qy * g.sh, px = x0 - qx * g.sw;
  int64_t off = (int64_t)(py * g.sw + px) * g.plane_stride + (int64_t)qy * g.rstride + qx;
  if (off > INT32_MAX || off < INT32_MIN) throw std::runtime_error("tap offset overflows int32");
  return (int32_t)off;
}

Grid make_grid(int buf, int H, int W, int C, int sh, int sw, int oy, int ox, int Hq, int Wq, int cap, bool unit_major = false) {
  Grid g;
  g.buf = buf; g.H = H; g.W = W; g.C = C;
  g.sh = sh; g.sw = sw; g.oy = oy; g.ox = ox; g.Hq = Hq; g.Wq = Wq;
  if (unit_major) { g.ustride = (int64_t)Hq * Wq; g.rstride = Wq; }
  else            { g.ustride = Wq; g.rstride = (int64_t)cap * Wq; }
  g.plane_stride = (int64_t)cap * Hq * Wq;
  g.pixels = g.plane_stride * sh * sw;
  return g;
}

int pick_bn(int N) { return N > 256 ? 256 : N; }

struct Builder {
  const WeightMap& w;
  NetPlan plan;
  int cap;
  bool cond;
  std::string sa, sb;                  // conditioning scope suffixes
  int cond_cols = 0;

  Builder(const WeightMap& w_, int cap_, bool cond_) : w(w_), cap(cap_), cond(cond_) { plan.capacity = cap_; }

  int new_buf(Grid g) {
    g.buf = (int)plan.bufs.size();
    plan.bufs.push_back(g);
    return g.buf;
  }

  // Registers one conditioning site (main.py:139-159) with per-channel scale s: returns its column
  // offset in the conditioning table and adds s * (b_a + b_b) to `constant`.
  int add_cond_site(const std::string& scope, int C, const std::vector<double>& s, std::vector<double>* constant) {
    const auto& wa = get(w, scope + sa + "/w", (size_t)kEmb * C);
    const auto& ba = get(w, scope + sa + "/b", C);
    const auto& wb = get(w, scope + sb + "/w", (size_t)kEmb * C);
    const auto& bb = get(w, scope + sb + "/b", C);
    int off = cond_cols;
    cond_cols += C;
    pending.push_back({off, C, &wa, &wb, s});
    for (int c = 0; c < C; ++c) (*constant)[c] += s[c] * ((double)ba[c] + (double)bb[c]);
    return off;
  }

  struct Pending {
    int off, C;
    const std::vector<float>*wa, *wb;
    std::vector<double> s;
  };
  std::vector<Pending> pending;
  std::vector<std::pair<int, std::vector<double>>> cond_consts;

  void finish_cond() {
    CondTable& t = plan.cond;
    t.n_cols = cond_cols;
    t.Pa.assign((size_t)kEmb * cond_cols, 0.f);
    t.Pb.assign((size_t)kEmb * cond_cols, 0.f);
    t.c.assign(cond_cols, 0.f);
    for (const auto& p : pending)
      for (int i = 0; i < kEmb; ++i)
        for (int c = 0; c < p.C; ++c) {
          t.Pa[(size_t)i * cond_cols + p.off + c] = (float)((*p.wa)[(size_t)i * p.C + c] * p.s[c]);
          t.Pb[(size_t)i * cond_cols + p.off + c] = (float)((*p.wb)[(size_t)i * p.C + c] * p.s[c]);
        }
    for (const auto& cc : cond_consts)
      for (size_t c = 0; c < cc.second.size(); ++c) t.c[cc.first + c] = (float)cc.second[c];
  }

  // Fills the bias / embedding part of an epilogue for a site with scale s and offset o.
  void site_epilogue(const std::string& site_scope, int C, int Ho, int Wo, const std::vector<double>& s,
                     std::vector<double> constant, Epilogue* e) {
    if (cond) {
      int off = add_cond_site(site_scope, C, s, &constant);
      e->cond_off = off;
      cond_consts.push_back({off, constant});
      std::vector<double> T = cont_embed(w, site_scope + "_temb", Ho, C);
      std::vector<double> F = cont_embed(w, site_scope + "_femb", Wo, C);
      e->ttab16.resize((size_t)Ho * C);
      e->ftab16.resize((size_t)Wo * C);
      for (int i = 0; i < Ho; ++i)
        for (int c = 0; c < C; ++c) e->ttab16[(size_t)i * C + c] = f32_to_f16_bits((float)(T[(size_t)i * C + c] * s[c]));
      for (int j = 0; j < Wo; ++j)
        for (int c = 0; c < C; ++c) e->ftab16[(size_t)j * C + c] = f32_to_f16_bits((float)(F[(size_t)j * C + c] * s[c]));
      // one combined table (there is no L1 left for small tables on the GPU, so one L2 read beats two)
      e->tftab.resize((size_t)Ho * Wo * C);
      for (int i = 0; i < Ho; ++i)
        for (int j = 0; j < Wo; ++j)
          for (int c = 0; c < C; ++c)
            e->tftab[((size_t)i * Wo + j) * C + c] = (float)((T[(size_t)i * C + c] + F[(size_t)j * C + c]) * s[c]);
    } else {
      e->bias.resize(C);
      for (int c = 0; c < C; ++c) e->bias[c] = (float)constant[c];
    }
  }

  // Appends the k-blocks and packed weights of a (kh x kw) convolution tap set reading grid `src`
  // (A map `map`) with top/left pads (pt, pl); weights w[kh][kw][Cin][C] scaled per output channel.
  void add_conv_taps(GemmLayer* L, const Grid& src, int map, const std::vector<float>& wt, int kh, int kw,
                     int Cin, int C, int pt, int pl, const std::vector<double>& scale) {
    int k0 = (int)L->kb.size() * kTileK;
    L->a_rowlen[map] = Cin;
    int kadd = kh * kw * Cin;
    int Knew = k0 + kadd;
    // grow [N][K] -> [N][Knew]
    std::vector<uint16_t> nw((size_t)L->N * Knew, 0);
    for (int n = 0; n < L->N; ++n)
      for (int k = 0; k < k0; ++k) nw[(size_t)n * Knew + k] = L->w[(size_t)n * k0 + k];
    for (int i = 0; i < kh; ++i)
      for (int j = 0; j < kw; ++j) {
        int32_t off = tap_offset(src, i - pt, j - pl);
        for (int c0 = 0; c0 < Cin; c0 += kTileK) L->kb.push_back({off, (int16_t)map, (int16_t)c0});
        for (int c = 0; c < Cin; ++c)
          for (int n = 0; n < C; ++n) {
            double v = (double)wt[(((size_t)i * kw + j) * Cin + c) * C + n] * scale[n];
            nw[(size_t)n * Knew + k0 + (i * kw + j) * Cin + c] = f32_to_f16_bits((float)v);
          }
      }
    L->w.swap(nw);
    L->K = Knew;
  }

  // Stride-1 4 x 4 convolutions with 64 channels in and out can be executed by the row-walk kernel.
  static void mark_walk(GemmLayer* L, const BlockSpec& b, int Cin, int C, int pt, int pl) {
    if (b.kh != 4 || b.kw != 4 || b.sh != 1 || b.sw != 1 || Cin != 64 || C != 64) return;
    L->walk = 1;
    L->c_kh = b.kh; L->c_kw = b.kw; L->c_pt = pt; L->c_pl = pl;
  }

  // One residual block (both flavours).  x: input grid (buf < 0 when Cin = 1: raw spectrogram).
  // y: output grid (already allocated, laid out for its consumer).
  void add_block(const BlockSpec& b, const BlockGeom& g, const Grid& x, const Grid& y, int Hin_raw, int raw_oh) {
    const int C = b.C, Cin = g.Cin;
    Affine bn1 = fold_bn(w, b.scope + "_conv1", C);
    Affine bnA = fold_bn(w, b.scope + "_addition", C);
    const auto& w1 = get(w, b.scope + "_conv1/w", (size_t)b.kh * b.kw * Cin * C);
    const auto& w2 = get(w, b.scope + "_conv2/w", (size_t)b.kh * b.kw * C * C);
    const auto& b2 = get(w, b.scope + "_conv2/b", C);

    Grid h = make_grid(-1, g.Ho, g.Wo, C, 1, 1, 0, 0, g.Hq, g.Wq, cap);
    h.buf = new_buf(h);

    // ---- conv1 (no bias) + conditioning -> BN -> ReLU ----
    Epilogue e1;
    e1.relu = 1;
    site_epilogue(b.scope + "_conv1", C, g.Ho, g.Wo, bn1.s, bn1.o, &e1);
    double macs1 = (double)g.Ho * g.Wo * b.kh * b.kw * Cin * C;
    if (Cin == 1) {
      DirectLayer& D = plan.first;
      D.name = b.scope + "_conv1";
      D.kh = b.kh; D.kw = b.kw; D.sh = b.sh; D.sw = b.sw; D.pt = g.pt; D.pl = g.pl;
      D.Hin = Hin_raw; D.Win = g.W; D.raw_oh = raw_oh;
      D.Ho = g.Ho; D.Wo = g.Wo; D.N = C;
      D.w.resize((size_t)b.kh * b.kw * C);
      for (int t = 0; t < b.kh * b.kw; ++t)
        for (int n = 0; n < C; ++n) D.w[(size_t)t * C + n] = (float)((double)w1[(size_t)t * C + n] * bn1.s[n]);
      D.epi = e1;
      D.out = h;
      D.macs_per_unit = macs1;
    } else {
      GemmLayer L;
      L.name = b.scope + "_conv1";
      L.Hq = g.Hq; L.Wq = g.Wq; L.Ho = g.Ho; L.Wo = g.Wo;
      L.a_buf[0] = x.buf;
      L.N = C;
      add_conv_taps(&L, x, 0, w1, b.kh, b.kw, Cin, C, g.pt, g.pl, bn1.s);
      L.BN = pick_bn(L.N);
      L.epi = e1;
      L.out = h;
      L.macs_per_unit = macs1;
      mark_walk(&L, b, Cin, C, g.pt, g.pl);
      build_groups(&L);
      plan.gemm.push_back(std::move(L));
    }

    // ---- conv2 (+b) + conditioning + identity/transform -> BN -> ReLU ----
    GemmLayer L;
    L.name = b.scope + "_conv2";
    L.Hq = g.Hq; L.Wq = g.Wq; L.Ho = g.Ho; L.Wo = g.Wo;
    L.a_buf[0] = h.buf;
    L.N = C;
    add_conv_taps(&L, h, 0, w2, b.kh, b.kw, C, C, g.pt2, g.pl2, bnA.s);
    L.BN = pick_bn(L.N);
    L.macs_per_unit = (double)g.Ho * g.Wo * b.kh * b.kw * C * C;
    std::vector<double> constant(C);
    for (int c = 0; c < C; ++c) constant[c] = bnA.s[c] * (double)b2[c] + bnA.o[c];
    Epilogue e2;
    e2.relu = 1;
    if (Cin == C) {
      if (b.sh != 1 || b.sw != 1) throw std::runtime_error("identity path with stride");
      e2.res_buf = x.buf;
      e2.res_scale.resize(C);
      for (int c = 0; c < C; ++c) e2.res_scale[c] = (float)bnA.s[c];
    } else {
      const auto& wt = get(w, b.scope + "_transform/w", (size_t)Cin * C);
      const auto& bt = get(w, b.scope + "_transform/b", C);
      for (int c = 0; c < C; ++c) constant[c] += bnA.s[c] * (double)bt[c];
      if (Cin == 1) {
        e2.r1_vec.resize(C);
        for (int c = 0; c < C; ++c) e2.r1_vec[c] = (float)((double)wt[c] * bnA.s[c]);
        e2.r1_sh = b.sh; e2.r1_sw = b.sw; e2.raw_oh = raw_oh;
      } else {
        L.a_buf[1] = x.buf;
        add_conv_taps(&L, x, 1, wt, 1, 1, Cin, C, 0, 0, bnA.s);
      }
      L.macs_per_unit += (double)g.Ho * g.Wo * Cin * C;
    }
    site_epilogue(b.scope + "_conv2", C, g.Ho, g.Wo, bnA.s, constant, &e2);
    L.epi = e2;
    L.out = y;
    if (L.a_buf[1] < 0) mark_walk(&L, b, C, C, g.pt2, g.pl2);
    build_groups(&L);
    plan.gemm.push_back(std::move(L));
  }
};

std::vector<BlockGeom> block_geometry(const std::vector<BlockSpec>& blocks, int H, int W) {
  std::vector<BlockGeom> out;
  int Cin = 1;
  for (const auto& b : blocks) {
    BlockGeom g{};
    g.H = H; g.W = W; g.Cin = Cin;
    same_pads(H, b.kh, b.sh, &g.Ho, &g.pt, &g.pb);
    same_pads(W, b.kw, b.sw, &g.Wo, &g.pl, &g.pr);
    int o;
    same_pads(g.Ho, b.kh, 1, &o, &g.pt2, &g.pb2);
    same_pads(g.Wo, b.kw, 1, &o, &g.pl2, &g.pr2);
    g.Hq = g.Ho + std::max(g.pt2, g.pb2);
    g.Wq = g.Wo + std::max(g.pl2, g.pr2);
    if (Cin > 1) {
      int hx, wx;
      if (b.sh == 1 && b.sw == 1) {
        hx = H + std::max(g.pt, g.pb);
        wx = W + std::max(g.pl, g.pr);
      } else {
        hx = (H + g.pt + g.pb + b.sh - 1) / b.sh;
        wx = (W + g.pl + g.pr + b.sw - 1) / b.sw;
      }
      g.Hq = std::max(g.Hq, hx);
      g.Wq = std::max(g.Wq, wx);
    }
    out.push_back(g);
    H = g.Ho; W = g.Wo; Cin = b.C;
  }
  return out;
}

// Grid of the tensor entering block `i` (written by block i-1), laid out for block i's convolutions.
Grid input_grid(const BlockSpec& b, const BlockGeom& g, int cap) {
  if (b.sh == 1 && b.sw == 1) return make_grid(-1, g.H, g.W, g.Cin, 1, 1, 0, 0, g.Hq, g.Wq, cap);
  return make_grid(-1, g.H, g.W, g.Cin, b.sh, b.sw, g.pt, g.pl, g.Hq, g.Wq, cap);
}

void build_blocks(Builder* B, const std::vector<BlockSpec>& blocks, int H, int W, int Hin_raw, int raw_oh,
                  const Grid& final_out) {
  std::vector<BlockGeom> geo = block_geometry(blocks, H, W);
  Grid x;                                               // raw for block 0
  for (size_t i = 0; i < blocks.size(); ++i) {
    Grid y;
    if (i + 1 < blocks.size()) {
      y = input_grid(blocks[i + 1], geo[i + 1], B->cap);
    } else {
      y = final_out;
    }
    y.buf = B->new_buf(y);
    B->add_block(blocks[i], geo[i], x, y, Hin_raw, raw_oh);
    x = y;
  }
}

}  // namespace

void build_groups(GemmLayer* L) {
  // fraction of the non-zero packed weights that fell into the fp16 subnormal range (reported at load time)
  size_t nz = 0, sub = 0;
  for (uint16_t h : L->w) {
    if ((h & 0x7fffu) == 0) continue;
    ++nz;
    if ((h & 0x7c00u) == 0) ++sub;
  }
  L->subnormal_frac = nz ? (double)sub / (double)nz : 0.0;
  L->groups.clear();
  const int n = (int)L->kb.size();
  std::vector<char> used(n, 0);
  for (int a = 0; a < n; ++a) {
    if (used[a]) continue;
    KGroup g{};
    g.row_off = L->kb[a].row_off; g.map = L->kb[a].map; g.col = L->kb[a].col;
    g.ntaps = 0;
    // taps of the same source / channel chunk whose rows lie within 7 rows above the first one
    for (int b = a; b < n && g.ntaps < 4; ++b) {
      if (used[b] || L->kb[b].map != g.map || L->kb[b].col != g.col) continue;
      const int64_t d = (int64_t)L->kb[b].row_off - g.row_off;
      if (d < 0 || d > 7) continue;
      g.shift[g.ntaps] = (int16_t)d;
      g.bk[g.ntaps] = b;
      g.ntaps++;
      used[b] = 1;
    }
    L->groups.push_back(g);
  }
}

static std::string grid_json(const Grid& g) {
  char b[512];
  snprintf(b, sizeof b,
           "{\"buf\":%d,\"C\":%d,\"H\":%d,\"W\":%d,\"mode\":%d,\"sh\":%d,\"sw\":%d,\"oy\":%d,\"ox\":%d,\"Hq\":%d,"
           "\"Wq\":%d,\"rstride\":%lld,\"ustride\":%lld,\"plane_stride\":%lld,\"pixels\":%lld}",
           g.buf, g.C, g.H, g.W, g.mode, g.sh, g.sw, g.oy, g.ox, g.Hq, g.Wq, (long long)g.rstride, (long long)g.ustride,
           (long long)g.plane_stride, (long long)g.pixels);
  return b;
}

std::string plan_to_json(const NetPlan& p) {
  std::string s = "{\"capacity\":" + std::to_string(p.capacity) + ",\"pool_buf\":" + std::to_string(p.pool_buf) +
                  ",\"cond_cols\":" + std::to_string(p.cond.n_cols) + ",\"bufs\":[";
  for (size_t i = 0; i < p.bufs.size(); ++i) s += (i ? "," : "") + grid_json(p.bufs[i]);
  s += "],\"first\":{\"name\":\"" + p.first.name + "\",\"macs\":" + std::to_string(p.first.macs_per_unit) +
       ",\"out\":" + grid_json(p.first.out) + "},\"gemm\":[";
  for (size_t i = 0; i < p.gemm.size(); ++i) {
    const GemmLayer& L = p.gemm[i];
    char b[512];
    snprintf(b, sizeof b,
             "%s{\"name\":\"%s\",\"Hq\":%d,\"Wq\":%d,\"Ho\":%d,\"Wo\":%d,\"N\":%d,\"BN\":%d,\"K\":%d,\"a_buf\":[%d,%d],"
             "\"res_buf\":%d,\"cond_off\":%d,\"groups\":%d,\"macs\":%.1f,\"walk\":%d,\"out\":",
             i ? "," : "", L.name.c_str(), L.Hq, L.Wq, L.Ho, L.Wo, L.N, L.BN, L.K, L.a_buf[0], L.a_buf[1], L.epi.res_buf,
             L.epi.cond_off, (int)L.groups.size(), L.macs_per_unit, L.walk);
    s += b + grid_json(L.out) + "}";
  }
  s += "]}";
  return s;
}

NetPlan build_main_plan(const WeightMap& w, int variant, int capacity) {
  Builder B(w, capacity, true);
  if (variant == 0) { B.sa = "_noise_pos_emb"; B.sb = "_noise_neg_emb"; }
  else              { B.sa = "_noise_emb";     B.sb = "_clean_emb"; }
  std::vector<BlockSpec> blocks = {                      // main.py:221-229
      {"resblock1_1", 4, 4, 1, 1, 64},  {"resblock1_2", 4, 4, 1, 1, 64},
      {"resblock2_1", 4, 4, 2, 2, 128}, {"resblock2_2", 4, 4, 1, 1, 128},
      {"resblock3_1", 3, 3, 2, 2, 256}, {"resblock3_2", 3, 3, 1, 1, 256},
      {"resblock4_1", 3, 3, 2, 2, 512}, {"resblock4_2", 3, 3, 1, 1, 512}};
  // resblock4_2 writes [n][w][h][c] so that last_conv ([5,1] VALID) is a plain GEMM over K = 5*512
  Grid head_in;
  head_in.mode = 1; head_in.C = 512; head_in.H = 5; head_in.W = 26;
  head_in.pixels = (int64_t)capacity * 26 * 5;
  build_blocks(&B, blocks, kWinFrames, kBins, kWinFrames, -(kWinFrames / 2), head_in);
  B.finish_cond();
  NetPlan& P = B.plan;
  const int head_buf = P.gemm.back().out.buf;

  // last_conv -> BN -> ReLU (main.py:231-235)
  {
    Affine bn = fold_bn(w, "last_conv", 512);
    const auto& wc = get(w, "last_conv/w", (size_t)5 * 512 * 512);
    GemmLayer L;
    L.name = "last_conv";
    L.Hq = 1; L.Wq = 26; L.Ho = 1; L.Wo = 26;
    L.a_buf[0] = head_buf;
    L.a_rowlen[0] = 2560;
    L.N = 512; L.BN = 256; L.K = 2560;
    for (int k = 0; k < 2560; k += kTileK) L.kb.push_back({0, 0, (int16_t)k});
    L.w.resize((size_t)512 * 2560);
    for (int n = 0; n < 512; ++n)
      for (int k = 0; k < 2560; ++k)     // k = h * 512 + c ; w[h][0][c][n]
        L.w[(size_t)n * 2560 + k] = f32_to_f16_bits((float)((double)wc[(size_t)k * 512 + n] * bn.s[n]));
    L.epi.bias.resize(512);
    for (int n = 0; n < 512; ++n) L.epi.bias[n] = (float)bn.o[n];
    L.epi.relu = 1;
    Grid o = make_grid(-1, 1, 26, 512, 1, 1, 0, 0, 1, 26, capacity);
    o.buf = B.new_buf(o);
    L.out = o;
    L.macs_per_unit = 26.0 * 2560 * 512;
    build_groups(&L);
    P.gemm.push_back(std::move(L));
  }
  // flatten (f * 512 + c) -> last_dense -> + mixed_central (main.py:236-242)
  {
    const auto& wd = get(w, "last_dense/w", (size_t)13312 * kBins);
    const auto& bd = get(w, "last_dense/b", kBins);
    GemmLayer L;
    L.name = "last_dense";
    L.a_buf[0] = P.gemm.back().out.buf;
    L.a_rowlen[0] = 13312;
    L.N = 208; L.BN = 208; L.K = 13312;
    for (int k = 0; k < 13312; k += kTileK) L.kb.push_back({0, 0, (int16_t)k});
    L.w.assign((size_t)208 * 13312, 0);
    // last_dense is zero-initialised and trained with a small learning rate (main.py:238): real checkpoints may
    // hold values below the fp16 normal range (6.1e-5).  Every output column is therefore scaled by a power of
    // two that brings its largest weight into [0.5, 1) before the cast (exact in fp32), and the head epilogue
    // multiplies the accumulator by the inverse (epi.res_scale doubles as that per-column factor for the head).
    L.epi.res_scale.assign(208, 1.f);
    for (int n = 0; n < kBins; ++n) {
      float mx = 0.f;
      for (int k = 0; k < 13312; ++k) mx = std::max(mx, std::fabs(wd[(size_t)k * kBins + n]));
      int e = 0;
      if (mx > 0.f && std::isfinite(mx)) {
        std::frexp(mx, &e);                              // mx = m * 2^e, m in [0.5, 1)
        e = std::min(std::max(-e, -24), 40);             // scale 2^-e, bounded
      }
      const float sc = std::ldexp(1.f, e);
      L.epi.res_scale[n] = std::ldexp(1.f, -e);
      for (int k = 0; k < 13312; ++k) L.w[(size_t)n * 13312 + k] = f32_to_f16_bits(wd[(size_t)k * kBins + n] * sc);
    }
    L.epi.bias.assign(208, 0.f);
    for (int n = 0; n < kBins; ++n) L.epi.bias[n] = bd[n];
    L.epi.relu = 0;
    L.epi.head = 1;
    L.macs_per_unit = 13312.0 * kBins;
    build_groups(&L);
    P.gemm.push_back(std::move(L));
  }
  return P;
}

NetPlan build_tower_plan(const WeightMap& w, int capacity) {
  Builder B(w, capacity, false);
  std::vector<BlockSpec> blocks = {                      // main.py:192-197
      {"embedding/noise_resblock1_1", 8, 4, 3, 2, 64},  {"embedding/noise_resblock2_1", 8, 4, 3, 2, 128},
      {"embedding/noise_resblock3_1", 4, 4, 1, 1, 256}, {"embedding/noise_resblock4_1", 4, 4, 1, 2, 512}};
  Grid pool = make_grid(-1, 23, 26, 512, 1, 1, 0, 0, 23, 26, capacity, true);   // unit-major for mean_pool_kernel
  build_blocks(&B, blocks, kCtxFrames, kBins, kCtxFrames, 0, pool);
  B.plan.pool_buf = B.plan.gemm.back().out.buf;
  B.plan.pool_pixels = 23 * 26;
  return B.plan;
}

}  // namespace nhans
