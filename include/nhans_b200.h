/* libnhans_b200.so - C ABI of the B200-native N-HANS inference hot path.
 *
 * The reference (N-HANS/N-HANS) has no plugin / operator / FFI boundary: the hot path is TensorFlow ops
 * called from Python (`apply.py`).  This header is the boundary a maintainer would bind with ctypes in
 * place of those ops; every entry point names the reference code it replaces
 * (SN = N_HANS___Selective_Noise, SS = N_HANS___Source_Separation).  INTEGRATION.md shows the binding.
 *
 * Conventions: plain pointers and sizes only; all functions return 0 on success and a negative code on
 * error (nhans_last_error gives the text); no exceptions cross the ABI; the caller owns every host
 * buffer, the context owns device memory, its CUDA stream and the pre-packed weights.  One context per
 * GPU; a context is not thread-safe, distinct contexts are independent (drive each from its own thread).
 * There is no CPU fallback: without a usable CUDA device nhans_create fails.
 */
#ifndef NHANS_B200_H_
#define NHANS_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct nhans_ctx nhans_ctx;

#define NHANS_OK 0
#define NHANS_ERR_CUDA (-1)
#define NHANS_ERR_ARG (-2)
#define NHANS_ERR_STATE (-3)
#define NHANS_ERR_CONTEXT_TOO_SHORT (-4) /* a --pos/--neg clip yields < 200 STFT frames (SN/apply.py:381-386) */
#define NHANS_ERR_KERNEL (-5)

#define NHANS_VARIANT_SELECTIVE_NOISE 0 /* SN/main.py::model : ctx_a = --pos, ctx_b = --neg           */
#define NHANS_VARIANT_SEPARATOR 1       /* SS/main.py::model : ctx_a = --neg (interference), ctx_b = --pos (target) */

/* Context on CUDA device `device`.  win_capacity / row_capacity = windows / context rows processed per
 * network pass (activation buffers are sized for them); 0 selects the defaults (2048 / 32). */
int nhans_create(int device, int variant, int win_capacity, int row_capacity, nhans_ctx** out);
void nhans_destroy(nhans_ctx* ctx);
const char* nhans_last_error(const nhans_ctx* ctx); /* ctx may be NULL: error of the last failed nhans_create */

/* Replaces tf.train.Saver.restore (SN/apply.py:428-432): `n` float32 variables under their TF names
 * (SURVEY.md App. C) with TF layouts (conv HWIO, dense [in, out]).  The context copies and pre-packs
 * them (batch-norm folding, fp16 operand layout, cont_embed tables of SN/main.py:127-137). */
int nhans_load_weights(nhans_ctx* ctx, const char* const* names, const int64_t* sizes, const float* const* data, int n);

/* ---- stage-level entry points (host pointers in / out, synchronous) --------------------------------- */

/* handle_signals (SN/apply.py:142-163): out[out_offs[u] ...] = float32(pcm / (max|pcm| + 1e-6)) computed in
 * float64, trimmed to a whole number of frames when `trim` != 0.  out_offs [U+1] is written. */
int nhans_normalise(nhans_ctx* ctx, const int16_t* pcm, const int64_t* offs, int U, int trim, float* out,
                    int64_t* out_offs);

/* tf.signal.stft(400, 160, 400, periodic Hann) + log(|X| + 1e-5) + angle (SN/apply.py:368-375) of U clips
 * pcm[offs[u] : offs[u+1]].  Writes frame_offs [U+1] (clip u has 1 + (N_u - 400) / 160 frames, 0 when
 * N_u < 400), and, when non-NULL, logmag / phase rows [frame_offs[U]][201] and peak [U].  Call with
 * logmag = phase = NULL first to size the outputs. */
int nhans_stft(nhans_ctx* ctx, const int16_t* pcm, const int64_t* offs, int U, float* logmag, float* phase,
               int64_t* frame_offs, int32_t* peak);

/* The same transform of float32 samples that are already normalised / mixed (apply_demo, SN/apply.py:241-251:
 * the on-the-fly mixture and the scaled noise signals returned by combine_signals).  No peak normalisation. */
int nhans_stft_f32(nhans_ctx* ctx, const float* x, const int64_t* offs, int U, float* logmag, float* phase,
                   int64_t* frame_offs);

/* Per-frame evaluation loss of the model graph (SN/main.py:243-246, SS/main.py:256-258):
 * example_loss[i] = mean_k( (denoised[i][k] - target[i][k])^2 * linspace(2, 1, 201)[k] ), rows of 201 bins. */
int nhans_eval_loss(nhans_ctx* ctx, const float* denoised, const float* target, int64_t n_frames, float* example_loss);

/* Embedding tower (SN/main.py:189-202): ctx_logmag [R][200][201] -> emb [R][512]. */
int nhans_embed(nhans_ctx* ctx, const float* ctx_logmag, int R, float* emb);

/* strided_crop(35, 1) + resnet blocks + head (SN/apply.py:378, 440-450; SN/main.py:218-242) without ever
 * materialising the windows: logmag rows [frame_offs[U]][201], one window per frame;
 * emb_a / emb_b [U][512]; denoised [frame_offs[U]][201] ('add_72:0'). */
int nhans_masknet(nhans_ctx* ctx, const float* logmag, const int64_t* frame_offs, int U, const float* emb_a,
                  const float* emb_b, float* denoised);

/* recover_samples_from_spectrum (SN/apply.py:189-201): exp, phasor, tf.signal.inverse_stft with
 * inverse_stft_window_fn(160, hann).  out_offs [U+1] is written (clip u has (T_u - 1) * 160 + 400 samples).
 * wav_f32 (reference output format) and / or wav_i16 = round(clip(y * (peak + 1e-6))) may be NULL;
 * peak may be NULL only when wav_i16 is NULL. */
int nhans_istft(nhans_ctx* ctx, const float* logmag, const float* phase, const int64_t* frame_offs, int U,
                const int32_t* peak, float* wav_f32, int16_t* wav_i16, int64_t* out_offs);

/* ---- fused end-to-end path: what apply_snc / apply_separator and the benchmark call ------------------ */

/* The same path for FLOAT clips that are already normalised / mixed on the host, fused on the device: apply_demo
 * (SN/apply.py:212-337, SS/apply.py:179-285: the on-the-fly mixture and the scaled context signals of combine_signals) and
 * stereo files of apply_snc / apply_separator (float64 channel mean, SN/apply.py:46-53).  Contexts are the first 200 STFT
 * frames of ctx_a / ctx_b (ctx_a may be NULL for the selective-noise variant: Silent.wav); the mask network runs over
 * mixture frames [start_frame, T_u) of every utterance (0 = apply_snc, 200 = apply_demo, SN/apply.py:251-262), the slice
 * zero padded like a whole utterance.  out_offs [U+1] is written ((T_u - start_frame - 1) * 160 + 400 samples each); call with
 * out_f32 = mixproc_f32 = NULL first to size the outputs ('mixed_demo.wav' / 'mixed_processed.wav' = mixproc).  Synchronous. */
int nhans_enhance_f32(nhans_ctx* ctx, const float* mix, const int64_t* mix_offs, int U, const float* ctx_a, const int64_t* a_offs,
                      const float* ctx_b, const int64_t* b_offs, int start_frame, float* out_f32, float* mixproc_f32,
                      int64_t* out_offs);

/* Output sizes for a batch: out_offs [U+1] in samples (trimmed lengths), without touching the GPU. */
int nhans_output_offsets(const int64_t* mix_offs, int U, int64_t* out_offs);

/* apply_snc (SN/apply.py:339-457) / apply_separator (SS/apply.py:288-397) for U utterances at once.
 * ctx_a may be NULL for the selective-noise variant: the all-zero Silent.wav context of apply_denoiser
 * (SN/apply.py:478-481).  Enqueues H2D copies, every kernel and D2H copies on the context stream and
 * returns; buffers must stay alive until nhans_sync.  Pinned host memory (nhans_host_alloc) makes the
 * copies asynchronous.  out_i16 / out_f32 / mixproc_f32 ('mixed_processed.wav', SN/apply.py:457-458) may
 * be NULL. */
int nhans_enhance_batch(nhans_ctx* ctx, const int16_t* mix, const int64_t* mix_offs, int U, const int16_t* ctx_a,
                        const int64_t* a_offs, const int16_t* ctx_b, const int64_t* b_offs, int16_t* out_i16,
                        float* out_f32, float* mixproc_f32);
int nhans_sync(nhans_ctx* ctx);
/* Consecutive nhans_enhance_batch calls are double buffered: the host-to-device copies of batch i + 1 and the
 * device-to-host copies of batch i - 1 run on their own CUDA streams while batch i computes (SN/apply.py:440-450 is
 * the loop this pipelines).  nhans_sync waits for everything; nhans_sync_previous waits only until the results of
 * every batch but the most recently enqueued one are in host memory, so a caller can unpack batch i while batch
 * i + 1 runs. */
int nhans_sync_previous(nhans_ctx* ctx);

/* The same path split at the PCIe boundary, for device-resident timing: upload stages a batch in HBM,
 * run processes the staged batch (no host traffic), download copies the results out. */
int nhans_upload(nhans_ctx* ctx, const int16_t* mix, const int64_t* mix_offs, int U, const int16_t* ctx_a,
                 const int64_t* a_offs, const int16_t* ctx_b, const int64_t* b_offs);
int nhans_run(nhans_ctx* ctx);
int nhans_download(nhans_ctx* ctx, int16_t* out_i16, float* out_f32, float* mixproc_f32);

/* Post-mix outputs of apply_snc for the batch nhans_run just processed (SN/apply.py:456-472), computed on the GPU
 * in one fused pass: mixed_processed = iSTFT(input spectrum), removed = mixed_processed - denoised,
 * snr_est[u] = mean(denoised^2) / mean(removed^2), compensated = denoised + removed * (ac ? snr_est / 20 : compensate).
 * A clip without frames (fewer than 400 samples), or whose removed signal is all zero, has snr_est = +inf; the --ac factor
 * is then 0, and a clip without frames has empty outputs.  Any output may be NULL; copies are enqueued on the context
 * stream (nhans_sync). */
int nhans_postmix(nhans_ctx* ctx, float compensate, int ac, float* mixed_f32, float* removed_f32, float* compensated_f32,
                  float* snr_est);

/* ---- streaming: live int16 mono streams, bit-identical to the batch path --------------------------------
 *
 * A stream is enhanced chunk by chunk as its samples arrive.  For every chunking, the concatenation of what a stream
 * emits equals the int16 / float32 output of nhans_enhance_batch for the whole clip bit for bit, given the same peak
 * and contexts.  Emission rule: after a stream has received N samples in all, F = 1 + (N - 400) / 160 frames (0 when
 * N < 400), it has emitted 160 * max(0, F - 17) samples; after its final step it has emitted (F - 1) * 160 + 400 (0 when
 * F = 0), what the batch path returns for the clip (trailing samples that fill no frame are dropped).  A window needs
 * the 17 frames after its centre and a 400-sample frame, so the algorithmic latency is 16 * 160 + 400 = 2960 samples
 * (185 ms at 16 kHz), plus up to 159 samples waiting for the next hop boundary.  nhans_stream_step_post also streams
 * the post-mix outputs of nhans_postmix (ac = 0), bit for bit, with a running snr_est.
 * nhans_load_weights closes every open stream.  Without loaded weights the calls below return NHANS_ERR_STATE. */

/* Opens n streams (one tower pass for all of them).  Stream i is conditioned on ctx_b[b_offs[i] : b_offs[i+1]] and
 * ctx_a[a_offs[i] : a_offs[i+1]], with the rules of nhans_enhance_batch (ctx_a may be NULL for the selective-noise
 * variant: Silent.wav; each clip must yield 200 frames, else NHANS_ERR_CONTEXT_TOO_SHORT).  peak[i] >= 0 replaces the
 * whole-clip max|x| of SN/apply.py:150, which a live stream cannot know: pass the peak nhans_stft reports for the whole
 * clip for output identical to the batch path, or a fixed full-scale value such as 32767.  It scales the input and the
 * int16 output.  ids [n] receives the stream ids.  Synchronous. */
int nhans_stream_open(nhans_ctx* ctx, int n, const int16_t* ctx_a, const int64_t* a_offs, const int16_t* ctx_b,
                      const int64_t* b_offs, const int32_t* peak, int* ids);
/* Appends chunk pcm[offs[i] : offs[i+1]] (any length, 0 included) to stream ids[i] (i < n, ids distinct) and processes
 * every window that has become computable across the n streams in the same network passes.  out_offs [n+1] is written
 * (offsets relative to out_offs[0] = 0); out_i16 / out_f32 (either may be NULL) receive each stream's newly emitted
 * samples there.  final may be NULL; final[i] != 0 flushes stream i, which then takes no further step.  An unknown or
 * closed id, an id given twice or a step after the final one is NHANS_ERR_ARG.  Synchronous; leaves the results of a
 * batch in flight (nhans_upload / nhans_run / nhans_download / nhans_postmix) untouched. */
int nhans_stream_step(nhans_ctx* ctx, int n, const int* ids, const int16_t* pcm, const int64_t* offs, const int* final,
                      int16_t* out_i16, float* out_f32, int64_t* out_offs);
/* nhans_stream_step plus the post-mix outputs of nhans_postmix (SN/apply.py:456-470) for the same samples: the same
 * arguments, checks, emission rule and out_offs, and mixed_f32 ('mixed_processed'), removed_f32 and compensated_f32 =
 * denoised + removed * compensate[i], each bit-identical to nhans_postmix(compensate[i], ac = 0) of the whole clip.
 * compensate [n] holds one factor per stream (NULL: 0; a non-finite factor counts as 0).  Every output array may be NULL.
 * snr_est [n] (may be NULL) receives each stream's running estimate: sum(denoised^2) / sum(removed^2) in float64 over every
 * sample the stream has emitted through nhans_stream_step_post (samples of plain nhans_stream_step calls do not count),
 * +inf while that removed energy is 0 (no sample yet, or a clip of fewer than 400 samples).  --ac has no streaming form: its
 * factor is the whole clip's snr_est, which only nhans_postmix knows.  Synchronous; leaves a batch in flight untouched. */
int nhans_stream_step_post(nhans_ctx* ctx, int n, const int* ids, const int16_t* pcm, const int64_t* offs, const int* final,
                           const float* compensate, int16_t* out_i16, float* out_f32, float* mixed_f32, float* removed_f32,
                           float* compensated_f32, int64_t* out_offs, float* snr_est);
/* Releases n streams, finalised or not. */
int nhans_stream_close(nhans_ctx* ctx, int n, const int* ids);
/* Host only (no context, no GPU): samples one step emits for a stream that goes from `before` to `after` samples
 * received (final != 0: its final step). */
int nhans_stream_emit_len(int64_t before, int64_t after, int final, int64_t* emitted);

/* Pinned host memory for the copies above. */
int nhans_host_alloc(int64_t bytes, void** out);
void nhans_host_free(void* p);

/* ---- measurement ---------------------------------------------------------------------------------- */

/* CUDA events on the context stream: record slot (0..15), elapsed between two recorded slots. */
int nhans_event_record(nhans_ctx* ctx, int slot);
int nhans_event_elapsed_ms(nhans_ctx* ctx, int start_slot, int stop_slot, double* ms);

/* Per-kernel statistics gathered with CUDA events around every launch while enabled (adds a few us per
 * launch).  kind: 0 tensor-core GEMM layers, 1 STFT, 2 iSTFT, 3 direct (Cin = 1) convolutions, 4 other;
 * stats [4] = {launches, total_ms, algorithmic_flops, algorithmic_bytes}.  kind 5: stats[0] = every kernel
 * this context launched since the last reset (counted whether or not profiling is enabled). */
int nhans_profile_enable(nhans_ctx* ctx, int on);
int nhans_profile_get(nhans_ctx* ctx, int kind, double* stats);
int nhans_profile_reset(nhans_ctx* ctx);
/* The same statistics for one tensor-core layer (net 0 main, 1 tower; layer = index into the plan's gemm list). */
int nhans_profile_get_layer(nhans_ctx* ctx, int net, int layer, double* stats);

/* ---- introspection (tests) -------------------------------------------------------------------------- */

/* JSON description of the layer plan (net 0 main, 1 tower): buffers, grids, layers.  Valid until the
 * next call on this context. */
const char* nhans_plan_json(nhans_ctx* ctx, int net);
/* Copy activation buffer `buf` of net (fp16 bits) to the host: n_elems must not exceed its size. */
int nhans_debug_read_buffer(nhans_ctx* ctx, int net, int buf, uint16_t* out, int64_t n_elems);
/* Debug: the spectra the fused path keeps in HBM for the batch nhans_run just processed (tests compare them with
 * the oracle's SN/apply.py:368-375 arrays): which 0 = log-magnitude [frames][201], 1 = unit phasors X / |X|
 * [frames][201][2] (the fused path stores phasors instead of angles), 2 = denoised log-magnitude [frames][201]. */
int nhans_debug_read_batch(nhans_ctx* ctx, int which, float* out, int64_t n_floats);
/* Debug (NHANS_DEBUG_TIMELINE=1 at create time): device timestamps of the last batches that went through
 * nhans_enhance_batch, in ms since the first one - out_ms[6 i + {0..5}] = H2D begin / end (copy-in stream), compute
 * begin / end, D2H begin / end (copy-out stream); -1 where a stage did not run.  Returns the number of batches written.
 * Synchronises the context. */
int nhans_debug_timeline(nhans_ctx* ctx, double* out_ms, int max_batches);
/* Debug: accumulated wait cycles of one tensor-core layer (needs NHANS_DEBUG_STATS=1 at create time):
 * {MMA waits accumulator free, MMA waits A, MMA waits B, epilogue waits accumulator ready, MMA warp total, ...}. */
int nhans_debug_layer_stats(nhans_ctx* ctx, int net, int layer, uint64_t* out8);
int nhans_device_info(nhans_ctx* ctx, int* sm_count, int* cc_major, int* cc_minor, int64_t* mem_bytes);

#ifdef __cplusplus
}
#endif
#endif /* NHANS_B200_H_ */
