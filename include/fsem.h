/*
 * fsem.h -- C ABI of libfsem_b200.so: batched PESQ and STOI/ESTOI scoring on sm_100a.
 *
 * The reference (kcoost/fast_speech_enhancement_metrics) is pure Python and has no
 * FFI layer of its own; this header is the boundary its two metric classes would bind
 * to replace their torch/torchaudio op chains:
 *
 *   fsem_pesq_*  replaces  PESQ.compute_metric / get_disturbances   (fast_se_metrics/PESQ.py:174-245)
 *                          incl. align_level (:92-102), pre_emphasize (:104-113),
 *                          get_bark_bands (:123-140), BarkFilterBank.forward (utils/bark.py:189-204),
 *                          Loudness.* (utils/loudness.py:48-67)
 *   fsem_stoi_*  replaces  BaseMetric.prepare_audio's resample (fast_se_metrics/base.py:16-21) and
 *                          STOI.compute_stoi / compute_metric         (fast_se_metrics/STOI.py:153-205)
 *                          incl. remove_silent_frames (:88-111), overlap_and_add (:71-86),
 *                          stft (:49-69), compute_segments (:121-127), equalize_clip (:129-139),
 *                          normalize (:113-119), compute_correlation (:141-151)
 *
 * Conventions
 *   - plain C types only; `stream` is a cudaStream_t passed as void*.
 *   - "device" pointers are CUDA device pointers owned by the caller; "host" pointers are
 *     ordinary (ideally pinned) host memory owned by the caller.  Inputs are never modified.
 *   - every call returns 0 on success and a negative FSEM_E_* code on failure;
 *     fsem_last_error() returns a thread-local message for the last failure.
 *   - device entry points are stream-ordered and do not synchronise; the *_host_* entry
 *     points include the host<->device copies and return after the scores are in host memory.
 *   - a context is bound to the CUDA device that was current when it was created and may
 *     be used from one host thread at a time.
 *   - arguments (designs, batch shapes, pointers) are checked before the first CUDA call, so a malformed
 *     argument gives FSEM_E_INVALID with or without a GPU.
 *   - there is no CPU fallback: without a CUDA device every call that gets past its argument checks fails
 *     with FSEM_E_CUDA.
 */
#ifndef FSEM_H_
#define FSEM_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define FSEM_API __attribute__((visibility("default")))
#else
#define FSEM_API
#endif

#define FSEM_VERSION 200 /* 0.2.0 */

#define FSEM_OK 0
#define FSEM_E_INVALID (-1) /* bad argument (null pointer, negative size, ...) */
#define FSEM_E_CUDA (-2)    /* CUDA runtime error (message in fsem_last_error) */
#define FSEM_E_WORKSPACE (-3) /* workspace too small */
#define FSEM_E_TOO_SHORT (-4) /* PESQ: fewer than 20 frames (reference: RuntimeError, PESQ.py:169) */

/* per-item status written next to the scores */
#define FSEM_ITEM_OK 0
#define FSEM_ITEM_TOO_SHORT 1 /* PESQ: < 20 frames; STOI: no 30-frame segment (score = NaN) */
#define FSEM_ITEM_NAN 2       /* score is NaN (e.g. all-zero PESQ input; reference gives NaN too) */

#define FSEM_PESQ_NBANDS 49
#define FSEM_PESQ_NFFT 512
#define FSEM_PESQ_HOP 256
#define FSEM_BP_SECTIONS 5
#define FSEM_STOI_NBANDS 15
#define FSEM_STOI_WIN 256
#define FSEM_STOI_HOP 128
#define FSEM_STOI_SEG 30

/* A batch of utterance pairs.  Rows are fp32, `stride` floats apart; row i holds
 * lengths[i] valid samples (all `n` when lengths == NULL).  Mirrors the
 * (clean_speech, denoised_speech) [batch, samples] tensors of BaseMetric.__call__
 * (base.py:41-43). */
typedef struct fsem_batch {
    const float* clean;     /* [batch, stride] */
    const float* deg;       /* [batch, stride] */
    const int32_t* lengths; /* [batch] or NULL; same memory space as clean/deg */
    int64_t batch;
    int64_t n;      /* samples per row (max length) */
    int64_t stride; /* row pitch in floats, >= n */
} fsem_batch_t;

/* Host-designed constants of PESQ.__init__ (PESQ.py:55-90, bark.py:129-164, loudness.py:42-46).
 * The 10th-order band-pass (scipy butter(5,[325,3250]) rounded to fp32, PESQ.py:80-81) is passed
 * in PARALLEL form: y = direct*x + sum_s (c0_s + c1_s z^-1) / (1 + a1_s z^-1 + a2_s z^-2) x,
 * obtained on the host from the poles/residues of the fp32-rounded polynomials. */
typedef struct fsem_pesq_design {
    float bp_direct;
    float bp_c0[FSEM_BP_SECTIONS];
    float bp_c1[FSEM_BP_SECTIONS];
    float bp_a1[FSEM_BP_SECTIONS];
    float bp_a2[FSEM_BP_SECTIONS];
    float pre_b[3];  /* pre-emphasis biquad numerator   (PESQ.py:85) */
    float pre_a[2];  /* a1, a2 of the denominator (a0 = 1) (PESQ.py:86) */
    float taper[15]; /* k/16, k = 1..15                 (PESQ.py:90) */
    int32_t warmup;  /* samples after which both IIR impulse responses are < fp32 eps */
    float hann[FSEM_PESQ_NFFT];              /* periodic Hann window (PESQ.py:63-71) */
    int32_t band_first_bin[FSEM_PESQ_NBANDS]; /* contiguous runs of FFT bins (bark.py:137-148) */
    int32_t band_num_bins[FSEM_PESQ_NBANDS];
    float pow_dens[FSEM_PESQ_NBANDS];  /* pow_dens_correction * Sp (bark.py:132) */
    float thresh[FSEM_PESQ_NBANDS];    /* absolute hearing threshold (loudness.py:43) */
    float zwicker_exp[FSEM_PESQ_NBANDS]; /* loudness exponents (loudness.py:45-46) */
    float width_bark[FSEM_PESQ_NBANDS];  /* band widths in Bark (bark.py:131) */
    float sl;                            /* Sl (loudness.py:25) */
    /* resample-on-ingest to 16 kHz (base.py:13,19-20): torchaudio sinc-Hann polyphase kernel, reduced rates;
     * rs_orig == rs_neu (e.g. both 1): input already is 16 kHz, rs_taps may be NULL */
    int32_t rs_orig, rs_neu, rs_width, rs_ntaps;
    const float* rs_taps; /* HOST pointer [rs_neu][rs_ntaps] */
} fsem_pesq_design_t;

/* Host-designed constants of STOI.__init__ (STOI.py:11-47) and of the ingest resampler
 * (base.py:13; torchaudio sinc_interp_hann kernel). */
typedef struct fsem_stoi_design {
    int32_t orig;   /* reduced input rate  (8 for 16 kHz -> 10 kHz); orig == neu: no resampling */
    int32_t neu;    /* reduced output rate (5) */
    int32_t width;  /* kernel half-width in input samples (10) */
    int32_t ntaps;  /* 2*width + orig (28) */
    const float* taps; /* HOST pointer, [neu][ntaps] fp32; may be NULL when orig == neu */
    float window[FSEM_STOI_WIN];       /* hann_window(257)[1:] exactly as torch builds it (STOI.py:24) */
    int32_t band_lo[FSEM_STOI_NBANDS]; /* third-octave band b sums FFT bins [lo, hi) (STOI.py:26-47) */
    int32_t band_hi[FSEM_STOI_NBANDS];
    float clip;      /* 1 + 10^(-beta/20) (STOI.py:137-138) */
    float dyn_range; /* 40 dB (STOI.py:22) */
} fsem_stoi_design_t;

typedef struct fsem_pesq_ctx fsem_pesq_ctx_t;
typedef struct fsem_stoi_ctx fsem_stoi_ctx_t;
typedef struct fsem_lsd_ctx fsem_lsd_ctx_t;
typedef struct fsem_resampler fsem_resampler_t;

FSEM_API int fsem_version(void);
FSEM_API const char* fsem_last_error(void);
/* number of kernel launches issued by this library on the calling thread since load */
FSEM_API int64_t fsem_launch_count(void);

/* Optional per-kernel timing (CUDA events on the launching stream).  Bench/diagnostics only,
 * process-global and not thread-safe.  fsem_profile_read synchronises on the recorded events and
 * returns the accumulated device time and launch count of kernel `index` (0 <= index < 15). */
FSEM_API int fsem_profile_enable(int on);
FSEM_API int fsem_profile_reset(void);
FSEM_API int fsem_profile_read(int index, const char** name, double* total_ms, int64_t* launches);

/* ------------------------------------------------------------------ PESQ */
FSEM_API int fsem_pesq_create(fsem_pesq_ctx_t** out, const fsem_pesq_design_t* design);
FSEM_API int fsem_pesq_destroy(fsem_pesq_ctx_t* ctx);
/* bytes of device workspace fsem_pesq_score_f32 needs for a [batch, n] call */
FSEM_API size_t fsem_pesq_workspace_bytes(const fsem_pesq_ctx_t* ctx, int64_t batch, int64_t n);
/* Device entry point.  mos_out[batch] fp32, status_out[batch] int32 (may be NULL): device. */
FSEM_API int fsem_pesq_score_f32(fsem_pesq_ctx_t* ctx, const fsem_batch_t* in, float* mos_out,
                        int32_t* status_out, void* workspace, size_t workspace_bytes, void* stream);
/* Host entry point: `in` holds HOST pointers; copies in chunks overlapped with compute,
 * scores land in host memory; synchronises before returning. */
FSEM_API int fsem_pesq_score_host_f32(fsem_pesq_ctx_t* ctx, const fsem_batch_t* in, float* mos_out,
                             int32_t* status_out);
/* Stage taps for parity tests (device pointers, after a score call on the same workspace):
 * copies the Bark-band power densities [2, batch, frames, 49] (clean then degraded, level-aligned:
 * the spectrum kernel applies g^2 = 1e7 * (n + 5120) * 1.04684 / power as it stores them) into `bark_out` and the
 * band-pass energies sum(y^2) [2, batch] (double) into `power_out`. */
FSEM_API int fsem_pesq_debug_taps(fsem_pesq_ctx_t* ctx, int64_t batch, int64_t n, const void* workspace,
                         float* bark_out, double* power_out, int64_t* frames_out, void* stream);

/* ------------------------------------------------------------------ STOI */
FSEM_API int fsem_stoi_create(fsem_stoi_ctx_t** out, const fsem_stoi_design_t* design);
FSEM_API int fsem_stoi_destroy(fsem_stoi_ctx_t* ctx);
FSEM_API size_t fsem_stoi_workspace_bytes(const fsem_stoi_ctx_t* ctx, int64_t batch, int64_t n);
/* Device entry point.  stoi_out/estoi_out[batch] fp32, kept_frames_out[batch] int32 (K, may be
 * NULL), status_out[batch] (may be NULL): device pointers. */
FSEM_API int fsem_stoi_score_f32(fsem_stoi_ctx_t* ctx, const fsem_batch_t* in, float* stoi_out,
                        float* estoi_out, int32_t* kept_frames_out, int32_t* status_out,
                        void* workspace, size_t workspace_bytes, void* stream);
FSEM_API int fsem_stoi_score_host_f32(fsem_stoi_ctx_t* ctx, const fsem_batch_t* in, float* stoi_out,
                             float* estoi_out, int32_t* kept_frames_out, int32_t* status_out);
/* Stage taps (device pointers, after a score call on the same workspace):
 * mask_out  [batch, mask_words] uint32 bit t of item i = frame t kept   (may be NULL)
 * tob_out   [2, batch, 15, tob_frames] third-octave magnitudes           (may be NULL)
 * resampled_out [2, batch, resampled_len] the 10 kHz signals             (may be NULL)
 * The three sizes are returned through dims_out[3] = {mask_words, tob_frames, resampled_len}. */
FSEM_API int fsem_stoi_debug_taps(fsem_stoi_ctx_t* ctx, int64_t batch, int64_t n, const void* workspace,
                         uint32_t* mask_out, float* tob_out, float* resampled_out,
                         int64_t* dims_out, void* stream);
/* Silent-frame decision margins (device pointers, after a score call on the same workspace and batch):
 * margin_out[batch] fp32 = min over the item's analysis frames of |(max_t E_t - dyn_range) - E_t| in dB, i.e. how
 * far the closest frame of the item is from flipping the bit-exact keep/drop decision of STOI.py:98-102
 * (+inf for an item without frames).  A batch whose smallest margin is above ~1e-4 dB cannot have been decided
 * differently by any fp32 evaluation order of the frame norm.  `lengths` as passed to the score call (or NULL). */
FSEM_API int fsem_stoi_mask_margin(fsem_stoi_ctx_t* ctx, int64_t batch, int64_t n, const int32_t* lengths,
                          const void* workspace, float* margin_out, void* stream);

/* ------------------------------------------------------------------ PESQ + STOI, one upload
 * Host entry point scoring BOTH metrics while copying every chunk of the batch host->device once
 * (callers of the reference always run both on the same tensors: README.md:29-30,
 * benchmark_metrics.py:22,24).  The STOI context must be built for the batch's sample rate.
 * Output arrays are HOST pointers; the *_status_out / kept_frames_out ones may be NULL. */
FSEM_API int fsem_pesq_stoi_score_host_f32(fsem_pesq_ctx_t* pesq, fsem_stoi_ctx_t* stoi, const fsem_batch_t* in,
                                  float* mos_out, int32_t* pesq_status_out, float* stoi_out, float* estoi_out,
                                  int32_t* kept_frames_out, int32_t* stoi_status_out);

/* Device entry point for both metrics (device pointers, separate workspaces sized by the two
 * *_workspace_bytes functions): the two complete kernel chains back to back on `stream`, each reading the
 * input itself; stream-ordered, no host synchronisation.  Results are identical to the two separate calls.
 * (Round 1 also carried a single-READ first-pass kernel and two-stream overlap modes behind an `overlap`
 * argument; both measured slower than this on B200 -- 9.5 ms against 4.0 + 3.5 ms for the two separate first
 * kernels, issue-bound rather than HBM-bound -- and were removed in 0.2.0.  DESIGN.md section 5.) */
FSEM_API int fsem_pesq_stoi_score_f32(fsem_pesq_ctx_t* pesq, fsem_stoi_ctx_t* stoi, const fsem_batch_t* in,
                             float* mos_out, int32_t* pesq_status_out, float* stoi_out, float* estoi_out,
                             int32_t* kept_frames_out, int32_t* stoi_status_out, void* ws_pesq, size_t ws_pesq_bytes,
                             void* ws_stoi, size_t ws_stoi_bytes, void* stream);

/* ------------------------------------------------------------------ ingest formats (SURVEY.md 8f rank 2)
 * The reference's boundary is float32 (base.py:16-21).  These entry points also take int16 PCM and fp16 sample
 * rows; samples are widened to fp32 with a value-preserving cast (no 1/32768 scaling -- both metrics are
 * scale-free), so the scores are bit-identical to scoring the same values as float32. */
#define FSEM_DTYPE_F32 0
#define FSEM_DTYPE_I16 1
#define FSEM_DTYPE_F16 2

/* Device entry points for any ingest dtype: exactly fsem_pesq_score_f32 / fsem_stoi_score_f32 /
 * fsem_pesq_stoi_score_f32 (which forward here with FSEM_DTYPE_F32), but `in->clean` / `in->deg` point at device rows of
 * `dtype` and `in->stride` counts ELEMENTS.  The first kernel of each chain (PESQ's IIR pass, STOI's resampler, or the
 * general resampler of a context that resamples on ingest) reads the rows in their own type, so a device-resident int16 /
 * fp16 batch is read from HBM once at 2 bytes per sample -- there is no widening pass.  (Only STOI on input that already
 * is 10 kHz has no such first kernel: it widens the rows into its workspace first.) */
FSEM_API int fsem_pesq_score(fsem_pesq_ctx_t* ctx, const fsem_batch_t* in, int dtype, float* mos_out, int32_t* status_out,
                    void* workspace, size_t workspace_bytes, void* stream);
FSEM_API int fsem_stoi_score(fsem_stoi_ctx_t* ctx, const fsem_batch_t* in, int dtype, float* stoi_out, float* estoi_out,
                    int32_t* kept_frames_out, int32_t* status_out, void* workspace, size_t workspace_bytes, void* stream);
FSEM_API int fsem_pesq_stoi_score(fsem_pesq_ctx_t* pesq, fsem_stoi_ctx_t* stoi, const fsem_batch_t* in, int dtype,
                         float* mos_out, int32_t* pesq_status_out, float* stoi_out, float* estoi_out,
                         int32_t* kept_frames_out, int32_t* stoi_status_out, void* ws_pesq, size_t ws_pesq_bytes,
                         void* ws_stoi, size_t ws_stoi_bytes, void* stream);

/* Device rows [rows, n] of `dtype` (pitch src_stride ELEMENTS) -> device fp32 rows (pitch dst_stride floats);
 * stream-ordered.  FSEM_DTYPE_F32 is a strided device-to-device copy. */
FSEM_API int fsem_ingest_f32(const void* src, int dtype, int64_t rows, int64_t n, int64_t src_stride, float* dst,
                    int64_t dst_stride, void* stream);

/* Host entry point for any ingest dtype and any subset of the two metrics: `pesq` or `stoi` may be NULL (that
 * metric is skipped and its output pointers are ignored).  clean / deg are HOST rows [batch, n] of `dtype` with
 * pitch `stride` elements (pinned memory for full PCIe speed), lengths [batch] HOST int32 or NULL.  Every chunk
 * crosses PCIe once at sizeof(dtype) bytes per sample and is scored in that dtype by the selected kernel chains
 * (fsem_pesq_score / fsem_stoi_score) while the next chunk is in flight.  With FSEM_DTYPE_F32 this is exactly fsem_pesq_score_host_f32 /
 * fsem_stoi_score_host_f32 / fsem_pesq_stoi_score_host_f32 (which forward here). */
FSEM_API int fsem_score_host(fsem_pesq_ctx_t* pesq, fsem_stoi_ctx_t* stoi, const void* clean, const void* deg, int dtype,
                    const int32_t* lengths, int64_t batch, int64_t n, int64_t stride, float* mos_out,
                    int32_t* pesq_status_out, float* stoi_out, float* estoi_out, int32_t* kept_frames_out,
                    int32_t* stoi_status_out);

/* ------------------------------------------------------------------ captured scoring (CUDA graph)
 * The reference scores a pair of tensors with ~100 eager torch ops per metric (PESQ.compute_metric, PESQ.py:232-245;
 * STOI.compute_metric, STOI.py:200-205); here a call is 3 + 7 kernel launches, and for the small batches of the
 * reference's README example (4 x 10 s) those launches run back to back at their latency floor.  fsem_graph_create
 * captures ONE scoring of fixed device buffers into a CUDA graph.  The batch is cut into `slices` contiguous parts
 * (<= 0: the library's choice, currently 1; at most 16) and every part's PESQ chain and STOI chain is a PARALLEL branch (they share
 * nothing but the read-only inputs): a replay costs one graph launch, small batches pay the longer of the two chains
 * instead of their sum, and for large batches the tail of every kernel overlaps with another branch's work.  Scores do
 * not depend on the slicing: they are bit-identical to fsem_pesq_stoi_score on the whole batch (the IIR time-chunk grid,
 * the only batch-dependent arithmetic, is planned for the whole batch).  Arguments as for fsem_pesq_stoi_score; `pesq`
 * or `stoi` may be NULL (that chain and its outputs are skipped).  The graph owns its workspaces and bakes in every
 * pointer: inputs and outputs must stay allocated, the caller rewrites the INPUT buffers in place between replays (the
 * static-buffer contract of CUDA graphs).  fsem_graph_launch is stream-ordered and does not synchronise; replays of one
 * graph must not overlap (they share the workspaces): launch them on one stream.  fsem_graph_nodes: kernel nodes per
 * replay; fsem_graph_slices: the slice count in use. */
typedef struct fsem_graph fsem_graph_t;
FSEM_API int fsem_graph_create(fsem_graph_t** out, fsem_pesq_ctx_t* pesq, fsem_stoi_ctx_t* stoi, const fsem_batch_t* in,
                      int dtype, float* mos_out, int32_t* pesq_status_out, float* stoi_out, float* estoi_out,
                      int32_t* kept_frames_out, int32_t* stoi_status_out, int slices);
FSEM_API int fsem_graph_launch(fsem_graph_t* g, void* stream);
FSEM_API int fsem_graph_nodes(const fsem_graph_t* g);
FSEM_API int fsem_graph_slices(const fsem_graph_t* g);
FSEM_API int fsem_graph_destroy(fsem_graph_t* g);

/* ------------------------------------------------------------------ resample-on-ingest (building block)
 * Replaces the torchaudio Resample of BaseMetric.prepare_audio (fast_se_metrics/base.py:13,19-20) for the metrics
 * that do not fuse it into their own first kernel (LSD, SDR): y[neu*k + p] = sum_j taps[p][j] * xpad[orig*k + j],
 * xpad = `width` zeros | x | zeros, output length ceil(neu * len / orig) per item.  `taps` is the HOST kernel
 * [neu][ntaps] torchaudio builds (design.sinc_hann_kernel), orig/neu the rates divided by their gcd.
 * fsem_resample_f32: `in` holds DEVICE rows; `out` is a DEVICE buffer [2, batch, out_stride] fp32 (clean rows, then
 * degraded rows); lengths_out[batch] (device int32) receives the per-item output lengths when in->lengths is given. */
FSEM_API int fsem_resampler_create(fsem_resampler_t** out, int32_t orig, int32_t neu, int32_t width, int32_t ntaps,
                          const float* taps);
FSEM_API int fsem_resampler_destroy(fsem_resampler_t* r);
FSEM_API int64_t fsem_resampled_len(const fsem_resampler_t* r, int64_t n);
FSEM_API int fsem_resample_f32(fsem_resampler_t* r, const fsem_batch_t* in, float* out, int64_t out_stride,
                      int32_t* lengths_out, void* stream);

/* ------------------------------------------------------------------ LSD (adjacent metric on the same FFT)
 * Replaces LSD.compute_metric (fast_se_metrics/LSD.py:33-52): scale-matched log-spectral distance on a
 * centred Hann-512/256 STFT.  `hann512` is the HOST window torch.hann_window(512) (LSD.py:16).
 * lsd_out[batch] fp32 and all batch pointers are DEVICE pointers; 16 kHz rows (other rates: fsem_resample_f32 first). */
FSEM_API int fsem_lsd_create(fsem_lsd_ctx_t** out, const float* hann512);
FSEM_API int fsem_lsd_destroy(fsem_lsd_ctx_t* ctx);
FSEM_API size_t fsem_lsd_workspace_bytes(const fsem_lsd_ctx_t* ctx, int64_t batch, int64_t n);
FSEM_API int fsem_lsd_score_f32(fsem_lsd_ctx_t* ctx, const fsem_batch_t* in, float* lsd_out, void* workspace,
                       size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------ SDR (adjacent metric)
 * Replaces SDR.compute_metric (fast_se_metrics/SDR.py:72-97; filter_length 512, no zero-mean, no diagonal
 * loading): unit-norm signals, 512 auto/cross-correlation lags, symmetric Toeplitz solve, coherence -> dB.
 * Stateless: no context.  sdr_out[batch] fp32 and all batch pointers are DEVICE pointers. */
FSEM_API size_t fsem_sdr_workspace_bytes(int64_t batch, int64_t n);
FSEM_API int fsem_sdr_score_f32(const fsem_batch_t* in, float* sdr_out, void* workspace, size_t workspace_bytes,
                       void* stream);

#ifdef __cplusplus
}
#endif
#endif /* FSEM_H_ */
