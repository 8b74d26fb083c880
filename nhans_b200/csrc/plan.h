// Layer plan of the N-HANS inference network for the B200 engine (host-only, no CUDA types).
//
// The network of N_HANS___Selective_Noise/main.py:98-242 (towers :189-216, residual stack :218-229,
// head :231-242) is lowered to two kinds of device layers:
//
//   * DirectLayer  - the Cin = 1 convolutions (resblock1_1_conv1, embedding/noise_resblock1_1_conv1)
//                    evaluated on CUDA cores straight from the fp32 log-magnitude spectrogram with
//                    the 35-frame window gather of SN/apply.py:170-186 done implicitly;
//   * GemmLayer    - every other convolution / dense layer as a "shifted-row GEMM"
//                        D[m, n] = sum_j  A_j[m + row_off_j, col_j : col_j + 64] . B[n, 64 j : 64 j + 64]
//                    over fp16 activations stored as padded pixel grids (see Grid below), so that a
//                    filter tap is a constant row offset and the A operand of every k-block is one
//                    plain 2-D TMA box.  Batch-norm, biases, the conditioning projections, the time /
//                    frequency embeddings, the residual add and ReLU are folded into the epilogue
//                    (SURVEY.md App. A.6).
//
// The same structures drive the CUDA engine (engine.cu) and the CPU plan interpreter used only by the
// tests (oracle/plan_exec.cc).
#pragma once

#include <cstdint>
#include <map>
#include <string>
#include <vector>

namespace nhans {

constexpr int kBins = 201;        // int(Fs*0.025)/2 + 1, SN/apply.py:409
constexpr int kWinFrames = 35;    // Mix_Win, SN/apply.py:38
constexpr int kCtxFrames = 200;   // Noise_Win, SN/apply.py:37
constexpr int kEmb = 512;
constexpr int kTileM = 128;
constexpr int kTileK = 64;

// An fp16 activation tensor [n][H][W][C] stored as a padded, optionally phase-split pixel grid:
// logical pixel (n, h, w) -> padded (y, x) = (h + oy, w + ox) -> phase plane (y % sh) * sw + (x % sw)
// at linear pixel plane * plane_stride + (y / sh) * rstride + n * ustride + (x / sw).
// Row-major over the image row first ("row-outer": rstride = cap * Wq, ustride = Wq): all units' copies of image
// row y are contiguous, so a vertical filter tap is the constant offset cap * Wq and the rows above the first /
// below the last image row of a plane are either outside the tensor (TMA zero-fills them) or the plane's spare
// rows (Hq - rows used).  A GEMM therefore only enumerates real output rows, no margin rows (they cost 5-17 % of
// the MMA work in a unit-major layout).  Horizontally a row segment holds W + pad pixels (shared left / right
// margin).  Everything that is not a logical pixel is zero for the lifetime of the buffer (it is never written),
// which is what implements the convolution padding.  The tower's final map uses the unit-major variant
// (ustride = Hq * Wq, rstride = Wq) because the pooling kernel wants a unit's pixels together; mode 1 is the
// head layout [n][w][h][c] read by last_conv as a plain GEMM.
struct Grid {
  int buf = -1;
  int C = 0;
  int H = 0, W = 0;
  int mode = 0;
  int sh = 1, sw = 1, oy = 0, ox = 0;
  int Hq = 1, Wq = 1;
  int64_t rstride = 1, ustride = 1; // pixels between image rows / between units
  int64_t plane_stride = 0;       // pixels between phase planes (= cap * Hq * Wq)
  int64_t pixels = 0;             // total pixels of the buffer (all planes)
};

inline int64_t grid_pixel(const Grid& g, int64_t n, int h, int w) {
  if (g.mode == 1) return (n * g.W + w) * g.H + h;
  int y = h + g.oy, x = w + g.ox;
  int plane = (y % g.sh) * g.sw + (x % g.sw);
  return plane * g.plane_stride + (int64_t)(y / g.sh) * g.rstride + n * g.ustride + (x / g.sw);
}

struct KBlock {                   // one 64-wide k-block of a GemmLayer
  int32_t row_off;                // pixel offset added to the tile's first row
  int16_t map;                    // 0: A0, 1: A1
  int16_t col;                    // first channel
  int16_t ho_lo, ho_hi;           // output rows [ho_lo, ho_hi) whose kernel row of this tap lies inside the source image;
                                  // for the other rows the tap reads only vertical padding (zeros)
};

// A group of up to 4 k-blocks whose A rows differ only by a small row shift (the kw taps of one kernel row
// and one 64-channel chunk): the engine loads ONE slab of 128 + 8 rows and feeds every tap from it through
// row-shifted UMMA descriptors, so A is fetched from L2 once per kernel row instead of once per tap.
// A tile of output row ho runs the group only if ho_lo <= ho < ho_hi (the union of its taps' ranges): for the
// other rows every A row the group reads is padding, so skipping it leaves every fp32 sum bit for bit the same.
struct KGroup {
  int32_t row_off;                // row offset of shift 0
  int16_t map;                    // 0: A0, 1: A1
  int16_t col;                    // first channel
  int16_t ntaps;
  uint8_t ho_lo, ho_hi;           // live output rows [ho_lo, ho_hi)
  int16_t shift[4];               // extra rows of tap t (0..7)
  int32_t bk[4];                  // k-block index of tap t in the packed weights
};

struct Epilogue {
  // v = acc + bias[utt * bias_stride + n] + tftab[ho * Wo + wo][n]
  //       + res_scale[n] * res[m][n] + r1_vec[n] * raw(n, ho, wo);  v = relu ? max(v, 0) : v
  int cond_off = -1;              // >= 0: per-utterance bias = column block of the conditioning table
  std::vector<float> bias;        // constant bias [N] (cond_off < 0)
  std::vector<float> tftab;       // [Ho * Wo][N]: time + frequency embedding (scaled), or empty
  std::vector<uint16_t> ttab16;   // the same embeddings kept separate in fp16, [Ho][C] and [Wo][C]: small enough
  std::vector<uint16_t> ftab16;   //   (~30 KB) to live in shared memory for the layers whose epilogue is the bottleneck
  int res_buf = -1;               // identity residual: buffer with the same row indexing
  std::vector<float> res_scale;   // [N]
  std::vector<float> r1_vec;      // rank-1 term on the raw spectrogram (1x1 transform with Cin = 1)
  int r1_sh = 1, r1_sw = 1;       // raw frame = win_frame[n] + ho * r1_sh + raw_oh, bin = wo * r1_sw
  int raw_oh = 0;
  int relu = 1;
  int head = 0;                   // 1: fp32 output [n][201] = acc * res_scale + bias + raw[center frame] (main.py:238-242;
                                  //    res_scale = inverse of the per-column power-of-two weight scale)
};

struct GemmLayer {
  std::string name;
  int Hq = 1, Wq = 1, Ho = 1, Wo = 1;     // compute space: m = (ho * cap + n) * Wq + wo, ho < Ho, valid wo < Wo (Hq: rows stored per plane)
  int a_buf[2] = {-1, -1};
  int a_rowlen[2] = {0, 0};               // elements per row of the 2-D view TMA reads (channels, or K for the head)
  int N = 0, BN = 0;                      // N padded to a multiple of 16; BN = columns per CTA tile
  int K = 0;                              // 64 * kb.size()
  std::vector<KBlock> kb;
  std::vector<KGroup> groups;             // kb regrouped for slab reuse (same k-blocks, same order of B)
  // [Ho]: the groups a tile of output row ho runs, as two index ranges s0 | e0 << 8 | s1 << 16 | e1 << 24 =
  // [s0, e0) + [s1, e1) (groups are ordered by kernel row, so the live conv groups are one range and the 1x1
  // transform groups, live for every row, the other)
  std::vector<uint32_t> row_groups;
  std::vector<uint16_t> w;                // fp16 bits, [N][K] (K contiguous)
  Epilogue epi;
  Grid out;                               // out.buf < 0 for the head
  double macs_per_unit = 0;               // algorithmic MACs per window / context row (SURVEY App. B)
  double exec_macs_per_unit = 0;          // the part of them the engine executes: k-blocks of live groups only
  // Row-walk eligible (conv_walk.cu): a stride-1 4 x 4 convolution with 64 channels in and out and no second A
  // source.  The k-blocks / weights above stay valid (plain N = 64 GEMM, what the CPU interpreter executes); the
  // engine repacks the weights as [kernel row block][cout] x [kw][cin] and walks the image rows instead.
  int walk = 0;
  int c_kh = 0, c_kw = 0, c_pt = 0, c_pl = 0;
  double subnormal_frac = 0;              // share of the non-zero fp16 weights that are subnormal (precision warning)
};

struct DirectLayer {
  std::string name;
  int kh = 0, kw = 0, sh = 1, sw = 1, pt = 0, pl = 0;
  int Hin = 0, Win = kBins, raw_oh = 0;   // input row r of unit n is raw frame win_frame[n] + r + raw_oh
  int Ho = 0, Wo = 0, N = 0;
  std::vector<float> w;                   // [kh*kw][N], BN scale folded
  Epilogue epi;
  Grid out;
  double macs_per_unit = 0;
};

struct CondTable {                        // bias_utt[u][j] = emb_a[u] . Pa[:, j] + emb_b[u] . Pb[:, j] + c[j]
  int n_cols = 0;
  std::vector<float> Pa, Pb;              // [512][n_cols]
  std::vector<float> c;                   // [n_cols]
};

struct NetPlan {
  int capacity = 0;                       // units (windows or context rows) the buffers are sized for
  std::vector<Grid> bufs;                 // one entry per activation buffer (geometry of its consumer)
  DirectLayer first;
  std::vector<GemmLayer> gemm;
  CondTable cond;                         // main net only
  int pool_buf = -1;                      // tower: buffer holding the final [n][23*26][512] map
  int pool_pixels = 0;
};

using WeightMap = std::map<std::string, std::vector<float>>;

struct ShapeMap {
  std::map<std::string, std::vector<int64_t>> s;
};

// variant 0: selective noise ('_noise_pos_emb' / '_noise_neg_emb'), 1: separator ('_noise_emb' / '_clean_emb')
NetPlan build_main_plan(const WeightMap& w, int variant, int capacity);
NetPlan build_tower_plan(const WeightMap& w, int capacity);

// TF 'SAME' padding: out = ceil(n / s), pad = max((out - 1) s + k - n, 0), before = pad / 2
void same_pads(int n, int k, int s, int* out, int* before, int* after);

// Regroups L->kb into L->groups and fills L->row_groups (call once the k-block list is complete).
void build_groups(GemmLayer* L);

// Split-K over ksplit consecutive slices of ceil(groups / ksplit) groups (gemm_tc.cu): does every slice run at least
// one group for every output row?  A slice that runs none would publish an accumulator no MMA has written.
bool every_split_live(const GemmLayer& L, int ksplit);

// JSON description of a plan (geometry only, no weights) for tests and DESIGN tables.
std::string plan_to_json(const NetPlan& p);

uint16_t f32_to_f16_bits(float f);
float f16_bits_to_f32(uint16_t h);

}  // namespace nhans
