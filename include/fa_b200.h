/*
 * fa_b200.h -- C-ABI of libfa_b200.so: the B200 (sm_100a) implementation of the formantanalyzer
 * feature-extraction hot path that tabahi/WebSpeechAnalyzer embeds.
 *
 * This is the drop-in boundary (SURVEY.md section 8(b)).  Everything the reference does between
 * "PCM arrives" and "callback(si, label, seg_time, features)" happens behind these calls:
 *
 *   reference interface (file:line, @B = byte offset in /root/reference/dist/main.js line 2)   entry point here
 *   ---------------------------------------------------------------------------------------   -----------------
 *   configure(cfg)                       @B3292   (used by /root/reference/src/index.js:393)   fa_config + fa_create
 *   reset_nodes / reset_segmentor        @B6992 / @B7303 -> reset_segmentation @B25053         fa_create / fa_reset
 *   LaunchAudioNodes(1, buf, cb, ...)    @B4469   (src/index.js:291)                           fa_submit_pcm + fa_run
 *   worklet "spectrum-processor" frames  @B6480 (un-vendored) -> spectrum_push @B30392         fa_run stage 1, fa_copy_spectrum / fa_copy_frames
 *   D()/O()/C() segmentor                @B25717 / @B27088 / @B28506                           fa_run stages 2-3, fa_copy_segments
 *   straighten_formants / sep_syllables  @B35074 / @B34757                                     fa_copy_formants / fa_copy_syllables
 *   formant_features / make_syl_features @B32369 / @B34407                                     fa_copy_features
 *   get_seg_timestamps / get_syls_timestamps @B31504 / @B31114                                 computed by the host shim from fa_segment / fa_syllable
 *   StopAudioNodes                       @B5699                                                fa_reset
 *
 * Rules: plain C types only; every call returns an fa_status (0 = ok, < 0 = error) and never
 * throws; a handle is not thread-safe, distinct handles are independent; there is no global
 * state and NO CPU FALLBACK: without a usable sm_100-class device fa_create fails with
 * FA_ERR_NO_DEVICE.
 */
#ifndef FA_B200_H_
#define FA_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define FA_API __attribute__((visibility("default")))
#else
#define FA_API
#endif

#define FA_N_FEATURES 53 /* /root/reference/src/localstore.js:7 (levels 5 and 13 -> 53) */
#define FA_N_CURVE_FEATURES 23 /* /root/reference/src/localstore.js:7 (level 12 -> 23): make_coeffs @B34527 */
#define FA_N_UTT_FEATURES 264 /* get_utterance_features, /root/reference/dist/main.js:2@B107983 (level 11) */
#define FA_ABI_VERSION 1
#define FA_ALL_UTTS (-1) /* utt_id of the getters: the whole batch, in submission order (utterance ids themselves are >= 0) */

typedef enum fa_status {
  FA_OK = 0,
  FA_ERR_INVALID_ARG = -1,
  FA_ERR_NO_DEVICE = -2,      /* no CUDA device / not sm_100 class; there is no CPU path */
  FA_ERR_CUDA = -3,           /* a CUDA runtime call failed; see fa_last_error */
  FA_ERR_NOT_RUN = -4,        /* results requested before fa_run + fa_sync */
  FA_ERR_UNKNOWN_UTT = -5,
  FA_ERR_CAPACITY = -6,       /* destination too small, or an internal table overflowed */
  FA_ERR_OUT_OF_MEMORY = -7,
  FA_ERR_BUSY = -8,           /* "Error: Already playing" (@B4469): fa_run while a run is in flight */
  FA_ERR_UNSUPPORTED = -9     /* e.g. an unknown output_level, fft size outside 256..16384 */
} fa_status;

/* spec_type (formantanalyzer defaults @B2972; tool-tips /root/reference/index.html:249-282) */
#define FA_SPEC_MEL 1
#define FA_SPEC_POWER 2
#define FA_SPEC_DFFT 3

/* element type of the spectrum rows (fa_config.spectrum_format).  F32: AnalyserNode.getFloatFrequencyData (dB, float32).
 * U8: AnalyserNode.getByteFrequencyData (W3C Web Audio API; SURVEY.md appendix B): trunc(clamp(255 / (max_db - min_db) *
 * (Y - min_db), 0, 255)) of the UNclamped dB value Y, -inf -> 0 -- a quarter of the bytes.  F16: the float view rounded to
 * IEEE half (clamp_db applies as for F32).  U8 / F16 rows are read with fa_copy_spectrum_raw / fa_set_spectrum_sink_raw. */
#define FA_SPECTRUM_F32 0
#define FA_SPECTRUM_U8 1
#define FA_SPECTRUM_F16 2

/* output_level (/root/reference/index.html:170-180) */
#define FA_LEVEL_BARS 1
#define FA_LEVEL_SPECTRUM 2
#define FA_LEVEL_SEGMENTS 3
#define FA_LEVEL_FORMANTS 4
#define FA_LEVEL_SEG_FEATURES 5
#define FA_LEVEL_SYL_FORMANTS 10
#define FA_LEVEL_UTTERANCE 11      /* "Utterance distributions": 264 doubles, cumulative, one row per stored segment */
#define FA_LEVEL_SYL_CURVES 12     /* "Syllable curves": 23 doubles per syllable (polynomial fits, numeric.uncmin) */
#define FA_LEVEL_SYL_FEATURES 13

typedef struct fa_config {
  /* ---- formantanalyzer fields (defaults @B2972) ---- */
  int32_t spec_type;        /* 1 */
  int32_t output_level;     /* 4 */
  int32_t plot_len;         /* 200 (only seg_limit_1 for levels <= 2 depends on it) */
  int32_t n_fft_bins;       /* 256 */
  int32_t n_mel_bins;       /* 128 */
  int32_t auto_noise_gate;  /* 1 */
  double f_min;             /* 50 Hz   */
  double f_max;             /* 4000 Hz */
  double window_width_ms;   /* 25 (informational: the analysis window is fft_size samples) */
  double window_step_ms;    /* 25 */
  double pause_length_ms;   /* 200 */
  double min_seg_length_ms; /* 50 */
  double voiced_max_db;     /* 100 */
  double voiced_min_db;     /* 10 */
  double pre_norm_gain;     /* 1000 */
  double high_f_emph;       /* 0 */
  /* ---- extension fields: the AnalyserNode front end that replaces the un-vendored worklet ---- */
  int32_t fft_size;         /* 2048 (power of two, 256..16384) */
  int32_t clamp_db;         /* 1: clamp the dB view to [min_db, max_db] */
  int32_t want_spectrum;    /* 1: materialise the dB spectrum [frames][fft_size/2] even for levels >= 3 */
  int32_t spectrum_format;  /* FA_SPECTRUM_F32 (0, default) | FA_SPECTRUM_U8 | FA_SPECTRUM_F16: element type of the spectrum rows */
  double smoothing;         /* smoothingTimeConstant 0.8 */
  double min_db;            /* -100 */
  double max_db;            /* -30 */
  double mag_scale;         /* 0 => fft_size (SURVEY.md finding 3) */
} fa_config;

typedef struct fa_segment {
  int32_t start;        /* seg_ci[si][0]: current_frame - len (reference quirk: late by the trailing pause) */
  int32_t len;          /* seg_ci[si][1] */
  int32_t stored;       /* index into the per-level stores (formants / features), -1 when the reference's
                           straighten_formants would have thrown and the segment was dropped (.catch -> L(-1)) */
  int32_t n_syllables;  /* levels 10/13 */
  int32_t first_syllable; /* index of its first syllable in the utterance's syllable table */
  int32_t row_offset;   /* first row of this segment in the utterance's formant table (rows of 9 floats) */
  double ymax;          /* adaptive maximum `y` at finalisation */
  double vmin;          /* adaptive minimum `v` at finalisation */
  double cs_ratio;      /* formant energy / non-formant energy (feature [2]) */
} fa_segment;

typedef struct fa_syllable {
  int32_t stored_seg;   /* index of the owning stored segment */
  int32_t start;        /* frame offset inside the segment */
  int32_t len;
  int32_t reserved;     /* level 12: 1 when the reference's make_coeffs threw at or before this syllable of the segment (its
                           row is NaN and was never handed to the callback), else 0 */
} fa_syllable;

/* Level 3 ("Segments"): the reference hands its callback the ranked formant tracks themselves (get_ranked_formants @B35670:
 * arrays of 18 fields, accumulate_fm @B35952).  Here: one fa_track per ranked track, in rank order, segment after segment, and
 * its points in time order.  The 18 fields of the reference's track array follow from the points (webspeechanalyzer_b200/api.py
 * track_arrays): [0] / [1] / [2] = [3] / [5] / [6] = lo / hi / frame / bin / amp of the LAST point, [4] the slope of the last
 * (up to four) bins, [7]..[12] the six point lists, [13] sum of the energies, [14] n_points, [15] sum of energy * bin, [16] 0,
 * [17] sum of (hi - lo + 1).  At level 3 fa_segment.n_syllables / first_syllable count and locate the segment's tracks,
 * fa_segment.row_offset its first point; fa_counts.syllables / formant_rows count the utterance's tracks / points. */
typedef struct fa_track {
  int32_t stored_seg;   /* index of the owning stored segment */
  int32_t first_point;  /* index of its first point in the utterance's point table */
  int32_t n_points;     /* [14] */
  int32_t reserved;
} fa_track;

typedef struct fa_track_point {
  int32_t frame;        /* [7]: the frame label c_ci inside the segment (the first one may be stale: quirk 1) */
  int16_t lo, hi, bin;  /* [8] [9] [10]: merged bounds and the loudest merged peak */
  int16_t reserved;
  uint32_t amp;         /* [11]: amplitude of the FIRST merged peak (quirk 8) */
  double energy;        /* [12]: sum of the frame over [lo, hi] (exact integer) */
} fa_track_point;

typedef struct fa_counts {
  int64_t samples;
  int32_t sample_rate;
  int32_t hop;            /* samples per frame step */
  int32_t frames;
  int32_t bands;          /* spec_bands */
  int32_t segments;       /* entries of seg_ci */
  int32_t stored_segments;
  int32_t formant_rows;   /* sum of len over stored segments */
  int32_t syllables;
  int32_t feature_rows;   /* level 5: stored segments; level 13: syllables */
  int32_t overflow;       /* non-zero if an internal table overflowed (results invalid) */
} fa_counts;

typedef struct fa_handle fa_handle;

FA_API void fa_config_default(fa_config* cfg);
FA_API int fa_abi_version(void);
FA_API const char* fa_status_string(int status);

FA_API int fa_create(const fa_config* cfg, int device, fa_handle** out);
FA_API int fa_destroy(fa_handle* h);
FA_API const char* fa_last_error(const fa_handle* h);
/* The configuration the handle was created with (spectrum rows hold fft_size / 2 values, level 11 rows 264 doubles, ...). */
FA_API int fa_get_config(const fa_handle* h, fa_config* out);

/* Use an externally owned cudaStream_t (e.g. torch's current stream); NULL restores the handle's own. */
FA_API int fa_set_stream(fa_handle* h, void* cuda_stream);

/* Stream for the spectrum-sink D2H copies (NULL restores the handle's own).  Handles that share one copy stream send their
 * dB rows back in submission order, one batch after the other, instead of interleaving on the PCIe link. */
FA_API int fa_set_d2h_stream(fa_handle* h, void* cuda_stream);

/* Number of sub-batches a run is split into (each on its own forked stream so that H2D, the kernels of different
 * sub-batches and the spectrum D2H overlap; at most 16): 0 = automatic, 1 = serial (per-stage timings are only defined then). */
FA_API int fa_set_pipeline(fa_handle* h, int n_sub_batches);

/* Caller-owned destination (ideally page-locked) for the dB spectrum rows of the whole batch, in submission order:
 * fa_run streams the rows into it as sub-batches finish; valid after fa_sync.  NULL removes the sink. */
FA_API int fa_set_spectrum_sink(fa_handle* h, float* dst, size_t cap_rows);
/* The same for any spectrum_format: rows of fft_size / 2 elements of the configured type (float32 / uint8 / half). */
FA_API int fa_set_spectrum_sink_raw(fa_handle* h, void* dst, size_t cap_rows);

/* Drop all submitted utterances and results (StopAudioNodes / a new batch). */
FA_API int fa_reset(fa_handle* h);

/* Copy one utterance of mono float32 PCM (host memory, owned by the caller) into the handle's
 * pinned staging buffer.  All utterances of one batch share sample_rate.  Returns its index. */
FA_API int fa_submit_pcm(fa_handle* h, int64_t utt_id, const float* pcm, size_t n_samples, int sample_rate);
FA_API int fa_submit_pcm_i16(fa_handle* h, int64_t utt_id, const int16_t* pcm, size_t n_samples, int sample_rate);
/* A whole batch in ONE caller buffer: utterance i is pcm[offsets[i] .. offsets[i+1]) and gets id first_utt_id + i.
 * If `pcm` is page-locked host memory (cudaHostAlloc / cudaHostRegister) the batch is NOT copied: the H2D transfer
 * reads the caller's buffer directly, which must then stay valid and unchanged until fa_sync.  Otherwise it is
 * staged like fa_submit_pcm.  Returns the index of the first utterance. */
FA_API int fa_submit_pcm_batch(fa_handle* h, int64_t first_utt_id, const float* pcm, const int64_t* offsets, int n_utt,
                               int sample_rate);

/* The same for 16-bit PCM (what a WAV file holds): with page-locked caller memory the int16 samples cross PCIe as they are
 * -- half the bytes of float32 -- and are converted on the device ((float)x * 2^-15, exact, identical to fa_submit_pcm_i16).
 * Pageable memory is converted on the host and staged like fa_submit_pcm_i16. */
FA_API int fa_submit_pcm_i16_batch(fa_handle* h, int64_t first_utt_id, const int16_t* pcm, const int64_t* offsets, int n_utt,
                                   int sample_rate);

/* The segmentor's own input, for callers that bring their own spectrum stage (e.g. frames captured from a browser
 * AnalyserNode / the reference's worklet): `n_frames` rows of `bands` uint32, one row per spectrum_push(frame, idx) of the
 * reference (/root/reference/dist/main.js:2@B30392).  `bands` must equal fa_spec_bands(cfg) -- the reference's own check,
 * same message ("Error: bins num mismatch").  The spectrum stage (K1a/K1b) is skipped for the batch; a batch holds
 * either PCM or frames (mixing fails with FA_ERR_INVALID_ARG); output_level must be >= 3.  The frames are copied (pinned
 * staging).  Returns the utterance index. */
FA_API int fa_submit_frames(fa_handle* h, int64_t utt_id, const uint32_t* frames, size_t n_frames, int bands);

/* Asynchronously: H2D copy of the staged PCM, stages 1-4 on the handle's stream, D2H of the result
 * tables.  fa_sync waits for it. */
FA_API int fa_run(fa_handle* h);
FA_API int fa_sync(fa_handle* h);

/* Device-resident variant for throughput measurement: upload once ... */
FA_API int fa_upload(fa_handle* h);
/* ... then run only the kernels on the resident PCM (no H2D, no D2H). */
FA_API int fa_run_resident(fa_handle* h);
/* and fetch the result tables of the last resident run to the host. */
FA_API int fa_download(fa_handle* h);

/* Per-stage device time of the last run in milliseconds (CUDA events on the handle's stream):
 * [0] spectrum, [1] peaks, [2] segment scan, [3] features, [4] whole run incl. copies. */
FA_API int fa_stage_times(fa_handle* h, float ms[5]);
/* The spectrum stage of the last run, kernel by kernel (its two launches): [0] frame-parallel FFT magnitudes |X|/N,
 * [1] smoothing recursion + dB view + band projection.  Like the stage times, only meaningful for a run with one sub-batch. */
FA_API int fa_spectrum_split_times(fa_handle* h, float ms[2]);
/* Number of kernel launches issued by the last run. */
FA_API int fa_launch_count(fa_handle* h);
/* Stream mode (utterances of >= 1000 frames on average): the smoothing recursion (stage 0) and the segmentor's control
 * scan (stage 1) run chunk-parallel from speculated entry states that a verification pass checks exactly; returns how many
 * chunks of that stage the last run had to redo (> 0 only means extra work, never a different result).
 * stage 2: utterances (epochs in stream mode) that the fast segment-scan kernel (<= 64 live tracks, <= 32 accepted peaks per
 * frame) handed back to the general kernel in the last run. */
FA_API int fa_stream_fixups(fa_handle* h, int stage);

FA_API int fa_num_utterances(const fa_handle* h);
FA_API int fa_result_counts(fa_handle* h, int64_t utt_id, fa_counts* out);
FA_API int fa_total_counts(fa_handle* h, fa_counts* out);
/* The fa_counts of every utterance of the batch, in submission order, in one call (a 100 k-utterance shard needs the rows per
 * utterance to key its dense feature table); returns the number of entries written. */
FA_API int fa_copy_counts_table(fa_handle* h, fa_counts* dst, size_t cap);

/* Caller-allocated destinations; `cap` counts elements of the destination type's row
 * (rows for tables).  Return value: rows written (>= 0) or an fa_status (< 0).  utt_id FA_ALL_UTTS returns the whole batch --
 * and FA_ERR_CAPACITY if ANY utterance of the batch overflowed an internal table (fa_counts.overflow; its tables are partial). */
FA_API int fa_copy_spectrum(fa_handle* h, int64_t utt_id, float* dst, size_t cap_rows);      /* rows of fft_size/2 dB values (FA_SPECTRUM_F32) */
FA_API int fa_copy_spectrum_raw(fa_handle* h, int64_t utt_id, void* dst, size_t cap_rows);   /* rows of fft_size/2 elements, any spectrum_format */
FA_API int fa_copy_frames(fa_handle* h, int64_t utt_id, uint32_t* dst, size_t cap_rows);     /* rows of `bands` uint32 */
/* Live streams (the reference fires its callback after every pause WHILE audio is still arriving, P() @B28869): the segmentor is
 * causal, so the segments that a PREFIX of the stream finalises on its own -- without segment_truncate @B30800, which only runs
 * when the source stops -- are exactly the ones the reference has called back by then.  fa_set_truncate(h, 0) switches the
 * final segment_truncate off for the following runs (default 1 = on): submit the stream so far, run, fire the callbacks of the
 * stores that are new; when the stream ends, run once more with truncation on.  (The whole prefix is re-analysed at every call:
 * at > 300 000 x real time that costs 0.2 ms per minute of audio.)  Host shim: webspeechanalyzer_b200/api.py LiveSession. */
FA_API int fa_set_truncate(fa_handle* h, int on);
FA_API int fa_copy_segments(fa_handle* h, int64_t utt_id, fa_segment* dst, size_t cap_rows);
FA_API int fa_copy_formants(fa_handle* h, int64_t utt_id, float* dst, size_t cap_rows);      /* rows of 9 float32 */
FA_API int fa_copy_energy(fa_handle* h, int64_t utt_id, float* dst, size_t cap_rows);        /* rows of 3 float32 */
FA_API int fa_copy_syllables(fa_handle* h, int64_t utt_id, fa_syllable* dst, size_t cap_rows);
FA_API int fa_copy_features(fa_handle* h, int64_t utt_id, double* dst, size_t cap_rows);     /* rows of 53 doubles */
/* Level 3 (P() @B28869 / O() @B27088, level-3 branches): the points of the ranked tracks; their fa_track headers come from
 * fa_copy_syllables (same 16-byte layout), fa_counts.syllables / formant_rows count tracks / points.  See fa_track. */
FA_API int fa_copy_track_points(fa_handle* h, int64_t utt_id, fa_track_point* dst, size_t cap_rows);
/* Level 11 (get_utterance_features @B107983, called from P() @B28869): rows of 264 doubles, one per stored segment of the
 * utterance, row k = the distribution over stores 0..k -- what the reference passes to its callback after store k; the
 * last row describes the whole utterance.  fa_counts.feature_rows counts these rows at level 11. */
FA_API int fa_copy_utterance_features(fa_handle* h, int64_t utt_id, double* dst, size_t cap_rows);
/* Level 12 (make_coeffs @B34527 -> polyfit @B33793 -> numeric.inv / uncmin): rows of 23 doubles, one per syllable, in syllable
 * order = [4th-degree fit of the energy in dB: 5 coefficients, residual, points | cubic fit of formant column 0: 4, residual,
 * points | cubic fit of column 3 | linear fit of column 6: 2, residual, points].  Where the reference's numeric would have
 * thrown, fa_syllable.reserved is 1 and the row is NaN (the reference's try / catch hands the rows made before the throw to
 * the callback and skips the rest of the segment).  fa_counts.feature_rows counts these rows at level 12. */
FA_API int fa_copy_curve_features(fa_handle* h, int64_t utt_id, double* dst, size_t cap_rows);

/* Stage-level taps for parity tests (candidate peaks of stage 2: packed lo | hi<<8 | pk<<16 | last<<24). */
/* ---- batched MLP inference on feature rows (the web app's emotion classifier; SURVEY.md 8(f) rank 3) -------------------
 * Replaces ml5 classifyMultiple on a tf.js Sequential of Dense layers (/root/reference/src/neuralmodel.js:540-585, models
 * under /root/reference/dist/nnmodel/<db>/cats_<label>/): kernels are row-major [in][out] float32 as in model.weights.bin,
 * inputs are min-max normalised with the ranges of model_meta.json ((x - min) / (max - min), in double, then float32).
 * fa_mlp_classify takes host rows (n_rows x dims[0] doubles) and writes n_rows x dims[n_layers] float32 outputs;
 * fa_mlp_classify_features classifies the feature rows of a finished handle where they are (device), one utterance
 * (utt_id >= 0) or the whole batch (utt_id < 0), and returns the number of rows.  No CPU path: FA_ERR_NO_DEVICE without a B200. */
#define FA_MLP_MAX_LAYERS 8
#define FA_MLP_LINEAR 0
#define FA_MLP_RELU 1
#define FA_MLP_SIGMOID 2
#define FA_MLP_SOFTMAX 3
typedef struct fa_mlp fa_mlp;
FA_API int fa_mlp_create(int n_layers, const int* dims /* n_layers + 1 */, const int* activations, const float* const* kernels,
                         const float* const* biases, const double* in_min, const double* in_max, int device, fa_mlp** out);
FA_API int fa_mlp_destroy(fa_mlp* m);
FA_API const char* fa_mlp_last_error(const fa_mlp* m);
FA_API int fa_mlp_classify(fa_mlp* m, const double* rows, size_t n_rows, float* probs);
FA_API int fa_mlp_classify_features(fa_mlp* m, fa_handle* h, int64_t utt_id, float* probs, size_t cap_rows);

/* ---- training of such a classifier on feature rows (K9, csrc/fa_train.cu; the algorithm is defined in DESIGN.md "K9") ----
 * Trains n_jobs independent models of one architecture (hidden layers linear / relu / sigmoid, softmax output, categorical
 * cross-entropy on integer labels) in one launch, without the host between steps.  The jobs share the row table `rows`
 * (n_rows x dims[0] doubles), its `labels` (int32 in [0, dims[n_layers])) and the options; job j trains on the row indices
 * row_idx[job_offsets[j] .. job_offsets[j + 1]) (repeats oversample, disjoint lists give folds), from its own seed and
 * initial parameters.  Parameter layout (init_params, out_params): per job, K7's -- for each layer the kernel [in][out],
 * then the bias, float32.  in_ranges NULL: each job's input ranges are the min / max of its own rows (a constant column
 * gets max = min + 1); otherwise [n_jobs][2][dims[0]] (min row, then max row) used as given.  out_ranges has that shape,
 * out_history is [n_jobs][epochs][2]: the row-weighted mean loss and the arg-max accuracy of every epoch.  Returns FA_OK,
 * FA_ERR_INVALID_ARG with a message in err (labels, indices, empty jobs, options, non-softmax output, non-finite values in
 * a selected row), FA_ERR_NO_DEVICE without an sm_100 device, or FA_ERR_CUDA / FA_ERR_OUT_OF_MEMORY. */
#define FA_OPT_SGD 0
#define FA_OPT_ADAM 1 /* beta1 0.9, beta2 0.999, epsilon 1e-7, bias-corrected (tf.js defaults) */
typedef struct fa_train_opts {
  double learning_rate;
  int optimizer;        /* FA_OPT_SGD / FA_OPT_ADAM */
  int epochs;           /* >= 0 */
  int batch_size;       /* >= 1; the last batch of an epoch holds the remaining rows and averages over them */
} fa_train_opts;
FA_API int fa_mlp_train(int n_layers, const int* dims /* n_layers + 1 */, const int* activations, const double* rows,
                        size_t n_rows, const int32_t* labels, int n_jobs, const int64_t* job_offsets /* n_jobs + 1 */,
                        const int32_t* row_idx, const uint64_t* seeds, const float* init_params, const double* in_ranges,
                        const fa_train_opts* opts, int device, float* out_params, double* out_ranges, double* out_history,
                        char* err, size_t err_cap);

FA_API int fa_copy_peak_candidates(fa_handle* h, int64_t utt_id, uint32_t* packed, int32_t* counts, size_t cap_rows,
                            int32_t* max_per_frame);

/* Stage-2 tap: g = sum e[1..B-1] of every frame (exact in double). */
FA_API int fa_copy_gsum(fa_handle* h, int64_t utt_id, double* dst, size_t cap_rows);

/* Host-side helpers that the shims share (no device needed). */
FA_API int fa_hop_samples(const fa_config* cfg, int sample_rate);
FA_API int fa_frames_for(const fa_config* cfg, int sample_rate, size_t n_samples);
FA_API int fa_spec_bands(const fa_config* cfg);

/* Page-locked host memory for callers that want the zero-copy paths (fa_submit_pcm*_batch, fa_set_spectrum_sink) without a
 * CUDA runtime of their own.  write_combined != 0: cudaHostAllocWriteCombined -- for buffers the host only WRITES (PCM on its
 * way to the device): not snooped during the PCIe transfer, very slow to read back on the host.  Portable across devices. */
FA_API void* fa_host_alloc(size_t bytes, int write_combined);
FA_API void fa_host_free(void* p);
/* Time `reps` back-to-back copies of `bytes` between `host` (page-locked) and a scratch buffer on `device` with CUDA events:
 * direction 0 = host to device, 1 = device to host.  The PCIe / host-memory floor of an end-to-end step, measured with the
 * caller's own buffer (bench.py runs it on all ranks at once). */
FA_API int fa_pcie_probe(int device, void* host, size_t bytes, int reps, int direction, float* ms_per_copy);

#ifdef __cplusplus
}
#endif
#endif /* FA_B200_H_ */
