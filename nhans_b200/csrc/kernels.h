// Device-side parameter blocks and kernel launchers of the engine.
#pragma once

#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace nhans {

// Per-unit (window / context row) lookup: frame row of the unit in the raw fp32 spectrogram, the
// [lo, hi) frame range of the clip it belongs to (rows outside read as 0.0, SN/apply.py:170-173) and
// the utterance index selecting the conditioning bias row.
struct UnitTable {
  const int* frame;
  const int* lo;
  const int* hi;
  const int* utt;
};

struct EpiDev {
  const float* bias;        // [n_utt or 1][bias_stride] (+ column offset already applied)
  int bias_stride;          // 0: one shared row
  const float* tftab;       // [Ho * Wo][N] time + frequency embedding, or null
  const __half* ttab16;     // fp16 [tab_H][C] / [tab_W][C] copies for the shared-memory-resident variant, or null
  const __half* ftab16;
  int tab_H, tab_W;
  const __half* res;        // identity residual rows [m][res_C] or null
  int res_C;
  const float* res_scale;   // [N]
  const float* r1_vec;      // [N] or null
  int r1_sh, r1_sw, raw_oh;
  const float* raw;         // fp32 spectrogram rows [frame][201]
  int relu;
  int head;                 // 1: out_f32[n][201] = acc + bias + raw[frame(n)]
  // output grid (plan.h Grid)
  __half* out;
  int out_C;
  int o_mode, o_sh, o_sw, o_oy, o_ox, o_H, o_W;
  long long o_plane, o_rstride, o_ustride;   // pixel = plane * o_plane + (y / sh) * o_rstride + unit * o_ustride + x / sw
  float* out_f32;
};

struct KGroupDev {            // plan.h KGroup
  int32_t row_off;
  int16_t map, col, ntaps, pad_;
  int16_t shift[4];
  int32_t bk[4];
};

struct GemmCfg {              // chosen by the host per layer shape
  int mt;                     // 128-row sub-tiles per CTA tile (256 / BN)
  int na, nb;                 // A slab ring / B tile ring depth
  int resident;               // all k-blocks of B fit in the ring: load once
  int il;                     // sub-tiles whose MMAs are interleaved (1 or 2; divides mt, <= na)
  int tab_bytes;              // > 0: the fp16 time / frequency tables are staged in shared memory
  int cta2;                   // 1: CTA pairs (cta_group::2): M = 256 MMAs, each CTA loads half of B
  int row;                    // 1: row-per-thread epilogue (no shared-memory transpose), see gemm_tc.cu
};

struct GemmDev {
  // compute space (plan.h): row m = ho * plane_pitch + unit * Wq + wo; only ho < Ho and rows < plane_rows of each
  // plane are enumerated: tile -> (chunk t, plane ho) with ho fastest, so that the kh taps of a pixel are read by
  // tiles that run close together in time (L2 reuse of the activations)
  int M;                    // rows enumerated = Ho * plane_rows
  int plane_pitch;          // capacity * Wq
  int plane_rows;           // units * Wq
  int N, BN;
  int num_kb;               // k-blocks (64 wide) of the packed weights
  int num_groups;
  const KGroupDev* groups;
  int Hq, Wq, Ho, Wo;
  UnitTable units;
  EpiDev epi;
  // split-K (head only: last_dense has 16 row tiles but K = 13312): tile -> (tile / ksplit, split = tile % ksplit),
  // split s accumulates the groups [s * gper, (s + 1) * gper) and stores its raw fp32 partial sums at
  // split_scratch[s][unit][N]; head_reduce_kernel adds them in a fixed order (deterministic) and applies the epilogue
  int ksplit;
  float* split_scratch;
  int* err_flag;
  unsigned long long* debug_stats;   // optional [8] cycle counters (wait times per role), or null
};

// Row-walk kernel (conv_walk.cu): stride-1 4 x 4 convolution, 64 -> 64 channels, over the compute space of GemmDev.
struct WalkDev {
  int plane_pitch;          // capacity * Wq
  int plane_rows;           // units * Wq
  int H, Wq, Wo;            // image rows (in = out), row segment pitch, valid pixels per segment
  int pt, pl;               // top / left padding
  UnitTable units;
  EpiDev epi;
  int* err_flag;
  unsigned long long* debug_stats;
  // Generated A operand (resblock1_1_conv2 only): instead of reading the first convolution's output from HBM, two
  // producer warps build every slab from the per-frame table of that convolution (FrameConvDev::C):
  // A[unit, r, x, :] = relu(C[variant(r)][frame(unit) + 34 utt(unit) - crow0 + r][x][:] + T1[r][:]) in fp16
  const float* gen_C;       // null: A comes from mapA (TMA)
  long long gen_crow0, gen_crow_cap;
  const __half* gen_ttab16; // [H][64] time embedding of the first convolution
};

struct DirectDev {
  int units;
  int kh, kw, sh, sw, pt, pl;
  int Hin, Win, raw_oh;
  int Ho, Wo, N;
  const float* w;           // [kh*kw][N]
  UnitTable units_tab;
  EpiDev epi;
};

constexpr int kGemmThreads = 352;     // A producer, B producer, MMA issuer, 8 epilogue warps
int gemm_smem_bytes(int BN, int num_kb, int tab_bytes, int cta2, int row, GemmCfg* cfg);
cudaError_t launch_gemm(cudaStream_t s, int n_sm, const CUtensorMap& mapA0, const CUtensorMap& mapA1,
                        const CUtensorMap& mapB, const CUtensorMap& mapBhalf, const GemmDev& p);
cudaError_t launch_direct_conv(cudaStream_t s, const DirectDev& p);
// mapA: the input grid as [pixels][64] (box 136 x 64), mapB: repacked weights [4 kernel-row blocks x 64][4 x 64] (box 256 x 64)
cudaError_t launch_walk(cudaStream_t s, int n_sm, const CUtensorMap& mapA, const CUtensorMap& mapB, const WalkDev& p);

// First convolution of the mask network, computed once per FRAME instead of once per (window, row): the 35-frame
// windows of one utterance are shifted copies of the same spectrogram, so conv(x)[window n, row h] depends only on
// the frame n - 17 + h - except for which kernel rows fall outside the window (rows h = 0, 33, 34), which gives four
// variants per frame.  frame_conv fills C[variant][crow][201][64] (fp32 FMA) for the frames a pass touches; crow =
// frame + 34 * utterance + row indexes the zero-extended utterance (17 virtual frames on either side), and the
// conditioning bias of the utterance and the frequency embedding F[w] are folded in (a C row belongs to one
// utterance).  window_expand then writes h1[n][h][w][:] = relu(C[variant(h)][crow(n) + h][w][:] + T[h]) in fp16:
// 35x fewer multiply-adds than the per-window kernel, what remains is the 1.8 GB store stream of a pass.
struct FrameConvDev {
  const float* raw;            // [frames][201] log-magnitude
  const long long* frame_offs; // [U + 1] device
  int u_first, u_last;         // utterances the pass touches
  long long crow0;             // first C row of the pass = first window + 34 * u_first
  int rows;                    // C rows to fill
  long long crow_cap;          // rows per variant plane of C
  const float* w;              // [16][64] taps (batch-norm scale folded)
  const float* bias;           // per-utterance bias rows (EpiDev::bias / bias_stride)
  int bias_stride;
  const __half* ftab16;        // [201][64] frequency embedding or null
  float* C;
};
cudaError_t launch_frame_conv(cudaStream_t s, const FrameConvDev& p);
// windows [unit0, unit1) of the pass
cudaError_t launch_window_expand(cudaStream_t s, const DirectDev& d, const float* C, long long crow0, long long crow_cap, int unit0,
                                 int unit1);

// bias_utt[u][j] = emb_a[u] . Pa[:, j] + emb_b[u] . Pb[:, j] + c[j]
// (stride 0 broadcasts one embedding row, e.g. the cached Silent.wav embedding of apply_denoiser)
cudaError_t launch_cond_table(cudaStream_t s, const float* emb_a, int stride_a, const float* emb_b, int stride_b, int U, const float* Pa,
                              const float* Pb, const float* c, int n_cols, float* out);
// emb[n][c] = mean over `pixels` rows of act[n][pixels][C]
cudaError_t launch_mean_pool(cudaStream_t s, const __half* act, int units, int pixels, int C, float* emb);
// out[n][c] = (sum_s scratch[s][n][c]) * scale[c] + bias[c] + raw[frame[n]][c], c < 201 (head of main.py:238-242)
cudaError_t launch_head_reduce(cudaStream_t s, const float* scratch, int ksplit, int units, int N, const float* scale, const float* bias,
                               const float* raw, const int* frame, float* out);
cudaError_t launch_units_main(cudaStream_t s, const long long* frame_offs, int U, int w0, int nwin, int* frame, int* lo,
                              int* hi, int* utt);
cudaError_t launch_units_rows(cudaStream_t s, int r0, int n, int rows_per_unit, int* frame, int* lo, int* hi, int* utt);

// ---- DSP ----
// peak[u] = max |pcm| per clip (int32; abs(-32768) wraps to -32768 like numpy int16, SN/apply.py:150)
cudaError_t launch_peaks(cudaStream_t s, const int16_t* pcm, const long long* offs, int U, int* peak);
// normalised float32 samples out[out_offs[u] + i] = f32(f64(pcm) / (peak + 1e-6)), i < out_offs[u+1] - out_offs[u]
cudaError_t launch_normalise(cudaStream_t s, const int16_t* pcm, const long long* offs, const long long* out_offs, int U,
                             const int* peak, float* out);
// frames, window, FFT-400, log(|X| + 1e-5), angle: logmag/phase rows [frame_offs[u] + t][201]
cudaError_t launch_stft(cudaStream_t s, const int16_t* pcm, const long long* offs, const long long* frame_offs, int U,
                        const int* peak, int max_frames_per_clip, float* logmag, float* phase,
                        bool phasor = false);   // phasor: `phase` receives unit phasors (float2 per bin) instead of angles
cudaError_t launch_eval_loss(cudaStream_t s, const float* den, const float* tgt, long long n, float* loss);
cudaError_t launch_stft_f32(cudaStream_t s, const float* x, const long long* offs, const long long* frame_offs, int U,
                            int max_frames_per_clip, float* logmag, float* phase, bool phasor = false);
// exp(logmag) * e^{j phase} -> irfft-400 -> synthesis window -> overlap-add -> f32 / int16 samples
cudaError_t launch_istft(cudaStream_t s, const float* logmag, const float* phase, const long long* frame_offs,
                         const long long* out_offs, int U, const int* peak, int max_frames_per_clip, float* out_f32,
                         int16_t* out_i16, bool phasor = false);
// apply_snc post-mix outputs (SN/apply.py:456-470): both iSTFTs, removed, energy sums; then compensated / snr_est
cudaError_t launch_istft_post(cudaStream_t s, const float* den_logmag, const float* mix_logmag, const float* phase,
                              const long long* frame_offs, const long long* out_offs, int U, int max_frames_per_clip,
                              float* den_f32, float* mixed_f32, float* removed_f32, double* sums, bool phasor = false);
cudaError_t launch_compensate(cudaStream_t s, const float* den, const float* removed, const long long* out_offs, int U,
                              const double* sums, float compensate, int ac, float* out, float* snr_est);
cudaError_t dsp_init_tables();

}  // namespace nhans
