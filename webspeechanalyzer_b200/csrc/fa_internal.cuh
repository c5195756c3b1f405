// fa_internal.cuh -- shared declarations of libfa_b200.so (sm_100a only; no CPU path).
//
// Stage map (SURVEY.md section 8(a)); @B = byte offset in /root/reference/dist/main.js line 2:
//   K1 fa_spectrum_*   S1 + S1b  AnalyserNode front end (replaces the un-vendored worklet @B6480) -> dB rows + uint32 band frames
//   K2 fa_peaks        S2        candidate peak scan of D() @B25863 (v-independent part)
//   K3 fa_segment      S2b/S3/S3b/S3c  D()/C()/O() @B25717/@B28506/@B27088, accumulate_fm @B35952, straighten @B35074, sep_syllables @B34757
//   K4 fa_features     S4        formant_features @B32369 + stats (src/stats.js:29-64)
//   K6 fa_utterance    (f)1      get_utterance_features @B107983 (level 11: 264-dim distributions)
//   K5 fa_compact      gathers the per-utterance tables into dense arrays for one D2H copy
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "fa_b200.h"

#define FA_MAX_BANDS 256

struct FaSpectrumParams {
  const float* pcm;              // concatenated utterances, each start 16-byte aligned, padded tail
  const long long* utt_off;      // [n_utt] first sample of utterance u
  const long long* utt_len;      // [n_utt] samples
  const long long* frame_off;    // [n_utt + 1] first frame row of utterance u
  int n_utt;                     // utterances of the whole batch (length of the tables above)
  int utt_begin, utt_count;      // the sub-batch this launch covers
  long long row_begin;           // first frame row of the sub-batch
  int hop, N, M, logM, B;
  const float* win;              // [N]
  const float2* tw;              // [M/2]   W_M^j
  const float2* tw_stage;        // [M-1]   stage-major: stage s (1-based) at offset 2^(s-1)-1, entries W_{2^s}^j
  const float2* ws;              // [M]     W_{2M}^k (mirror rule above M/2)
  const int* bm_k0;              // [B]
  const int* bm_cnt;             // [B]
  const int* bm_off;             // [B+1]
  const float* bm_w;             // [n_weights]
  int n_weights;
  const float* emph;             // [B]
  int use_emph, power;
  float gain, tau, omt, inv2N, min_db, max_db;
  int clamp_db;
  float* spec_db;                // [F_total][M]: |X|/N rows from K1a, converted to dB in place by K1b (fast path);
                                 // generic path: dB rows or nullptr
  int scratch_mag;               // 1: spec_db is allocated and may be used as the K1a -> K1b magnitude buffer
  int write_db;                  // 1: the caller wants the dB rows
  int k1a_variant;               // FA_K1A_VARIANT: launch shapes 1-3 (overlap experiments), 4 = sqrt.rn for every magnitude (A/B)
  int fused;                     // 1: fft_size 2048 in utterance mode runs the fused K1 kernel (no magnitude round trip)
  int spec_fmt;                  // FA_SPECTRUM_F32 / _U8 / _F16: element type of the rows the caller gets
  void* spec_q;                  // [F_total][M] uint8 or half rows (spec_fmt != F32); the magnitudes then stay in spec_db
  float byte_scale;              // 255 / (max_db - min_db)
  long long n_rows;              // frames of the sub-batch
  uint32_t* frames;              // [F_total][B] or nullptr
  int* work_counter;             // dynamic utterance queue
  // K1b stream mode (long utterances): the smoothing recursion is run per CHUNK of `chunk_frames` frames, every chunk but
  // the first from a SPECULATED entry state (a warm-up over the `warm_frames` frames before it, started from zero), and a
  // verification pass compares each chunk's true exit state with the next chunk's speculated entry bit for bit,
  // recomputing the (rare) chunks whose warm-up had not converged.  chunk_frames == 0: one pass per utterance.
  int chunk_frames, warm_frames;
  const int* chunk_utt;          // [n_chunks] work items of this launch: utterance ...
  const int* chunk_idx;          // ... and chunk inside it
  const long long* chunk_base;   // [n_utt + 1] first state slot of every utterance
  int n_chunks;
  float* st_entry;               // [total chunks][M]
  float* st_exit;                // [total chunks][M]
  float* spec_out;               // dB rows in stream mode (the magnitudes must survive until verified); nullptr: in place
  int* fixups;                   // chunks recomputed by the verification pass
};

// one candidate peak of a frame (K2 -> K3), 32 bytes = one DRAM sector
struct __align__(16) FaCand {
  uint32_t packed;               // lo | hi<<8 | pk<<16 | last<<24 (trimmed bounds)
  uint32_t amp;                  // e[pk]
  unsigned long long pl;         // P[lo - 1]  (P = inclusive prefix sums of the frame, exact)
  unsigned long long ph;         // P[hi]
  unsigned long long pad;
};

struct FaPeaksParams {
  const uint32_t* frames;        // [F_total][B]
  int B, maxp;
  long long n_frames;            // frames of the sub-batch
  long long row_begin;
  FaCand* cand;                  // [F_total][maxp]
  int* ncand;                    // [F_total]
  double* gsum;                  // [F_total] sum e[1..B-1]
};

// One finalisation of the control scan (K3a -> K3b), or of the utterance-mode scan (fa_segment2_kernel -> the finaliser): the
// frames of the track epoch that ends in it and the scalar state O() @B27088 reads.  Index in the per-utterance table = index
// in seg_ci.  The epoch's points sit in the point pool from (frame_off[u] + first) * maxp on.
struct __align__(16) FaEpoch {
  int first;                     // first frame of the epoch (frame index inside the utterance): tracks were cleared before it
  int last;                      // last frame to replay (the frame that triggered the finalisation; F - 1 for segment_truncate)
  int n_arg, no_fm_segs, current_frame, c_ci;
  int trk_off, trk_cap;          // the epoch's slice of the utterance's track table (capacity = accepted peaks of the epoch)
  double y, v;                   // thresholds at finalisation
  double c_energy, s_energy;     // utterance-mode scan only: the tracker's energies at finalisation
  int n_tr, n_pts;               // ... and its track / point counts (the control scan leaves them to K3b's replay)
};

// the control state that crosses a chunk boundary of the control scan (K3a stream mode)
struct __align__(8) FaCtlState {
  int c_started, no_fm_segs, c_ci, w, k, epoch_first;
  int n_epochs;                  // accepted finalisations inside the chunk
  int fired;                     // the gate's T/k reset fired inside the chunk
  int overflow, n_events;        // n_events: reset tests recorded for the chunk
  double y, v, x, v0, T;
};

struct FaSegmentParams {
  const FaCand* cand;            // [F_total][maxp]
  const int* ncand;
  const double* gsum;
  const long long* frame_off;    // [n_utt + 1]
  int n_utt, B, maxp, level;
  int utt_begin, utt_count;
  // reset_segmentation @B25053
  int max_voiced_bin, seg_min_frames, auto_gate;
  double seg_breaker, y0, v0;
  // workspaces (per utterance u: base index = frame_off[u] * K + const * u)
  int track_cap_mul, track_cap_add;   // tracks capacity of utterance u = F_u * mul + add
  long long* track_base;              // [n_utt + 1] prefix of capacities
  int* trk_count; double* trk_sum_e; double* trk_sum_eb; double* trk_mean; int* trk_order; int* trk_rank; signed char* trk_slot;
  // point pool: capacity F_u * maxp, base = frame_off[u] * maxp
  int* pt_track; int* pt_ord; int* pt_frame; int* pt_binspan; double* pt_e;   // binspan = bin | lo << 8 | (hi - lo + 1) << 16
  int* pt_amp;                        // level 3 only (else nullptr): amplitude of the point ([11] of the reference's track array)
  fa_track_point* track_points;       // level 3 only: exported points, base = frame_off[u] * maxp (and fa_track headers in `syls`
                                      // at the same base instead of frame_off[u] + u)
  int* row_count; int* row_off;       // [F_total + n_utt] scratch (per utterance F_u + 1)
  int* row_list;                      // [F_total * maxp]
  unsigned long long* cs_spill;       // [n_utt][6][128] candidate scores beyond the three kept in shared memory
  int finalize_in_smem;               // 1: segments that fit are finalised in shared memory (0 forces the HBM path: tests)
  int no_truncate;                    // 1: the utterances are prefixes of running streams: no segment_truncate @B30800 at their end
  // impl 2 (default): tracking with peak-lane ownership (accumulate_fm2: <= 64 live tracks, <= 32 accepted peaks per frame);
  // an utterance / epoch that needs more is flagged (overflow == 2) and redone by the general kernel (impl 1) in a second,
  // normally empty launch with redo_only = 1
  int impl, redo_only;
  int* redo_count;                    // utterances / epochs handed back to the general kernel (fa_stream_fixups(h, 2))
  int warps_per_cta, reg_cap;         // launch shape knobs (FA_K3_WARPS, FA_K3_REGS), read once per handle
  int smem_per_warp;                  // bytes of shared memory per warp (set by fa_launch_segment)
  // mode 1: control scan (K3a, warp per utterance) + epoch-parallel tracking / finalisation (K3b, warp per epoch) + fix-up (K3c)
  int mode;
  unsigned* fr_ctl;                   // [F_total] bit 31: the frame reaches accumulate_fm; low bits: its (stale) label c_ci
  double* fr_v;                       // [F_total] gate threshold v after the frame (= v at the start of the next frame)
  FaEpoch* epochs;                    // [F_total + n_utt] per-utterance tables at base frame_off[u] + u (mode 1, and the
                                      // finalisations fa_segment2_kernel records at every level but 3)
  int2* work;                         // epoch work list of this sub-batch: (utterance, seg_ci index)
  int* work_count;                    // [2]: entries in the list, next entry to take
  int n_workers;                      // warps of the K3b grid (cs_spill has one slice per worker in mode 1)
  // K3a chunked (long utterances): every chunk of `ctl_chunk` frames is scanned from a SPECULATED entry state (a warm-up over
  // the `ctl_warm` frames before it, from the initial state); a verification pass walks the chain, accepts a chunk when its
  // speculated entry equals the true exit of its predecessor (T, k up to a replay of the gate's tests) and rescans it otherwise
  int ctl_chunk, ctl_warm;
  const int* cchunk_utt; const int* cchunk_idx; const long long* cchunk_base; int n_cchunks;
  FaCtlState* ctl_entry; FaCtlState* ctl_exit;   // [total chunks]
  // the gate's reset tests of a chunk, in order, at [frame_off[u] + a + i]: T and k in front of the test (k bit 31: it fired)
  // and the threshold factor 30 v
  double* fr_T; int* fr_k; double* fr_thr;
  int* ctl_fixups;
  // outputs (per utterance tables at base frame_off[u] + u, capacity F_u + 1)
  fa_segment* segs; int* n_segs; int* n_stored;
  float* formants;                    // [F_total][9]   rows of utterance u start at frame_off[u]
  float* energy;                      // [F_total][3]
  int* n_rows;                        // [n_utt]
  fa_syllable* syls; int* n_syls;
  int* overflow;                      // [n_utt]
};

struct FaFeatureParams {
  const long long* frame_off;
  int n_utt, level;
  int utt_begin, utt_count;
  const fa_segment* segs; const int* n_segs;
  const fa_syllable* syls; const int* n_syls;
  const float* formants;
  int row_slices;                     // CTAs per utterance (grid.y): rows are dealt round-robin over slices x warps
  const FaEpoch* epochs;              // K3 stream mode: the rows of segment s sit at the epoch's first frame (not compacted);
                                      // nullptr: at fa_segment.row_offset
  double* features;                   // [(F_total + n_utt)][53] per-utterance rows at base frame_off[u] + u
  int* n_feat;                        // [n_utt]
};

// K8 (level 12): 23-dim polynomial-curve rows, one per syllable (fa_curves.cu)
struct FaCurveParams {
  const long long* frame_off;
  int n_utt;
  int utt_begin, utt_count;
  const fa_segment* segs; const int* n_segs;
  fa_syllable* syls; const int* n_syls;  // .reserved is set where the reference's make_coeffs would have thrown
  const float* formants; const float* energy;
  const FaEpoch* epochs;              // see FaFeatureParams
  int2* list; int* list_count;        // work list of this sub-batch: (utterance, syllable) pairs, and its length (zeroed per run)
  long long list_cap;                 // upper bound of the list length (frames / 2 + utterances of the sub-batch)
  double* work;                       // [F_total][34] powers / ordinates of the four fits of the syllable that owns the row
  int* status;                        // [(F_total + n_utt)][4] FA_CURVE_* of every fit
  double* rows;                       // [(F_total + n_utt)][23] per-utterance rows at base frame_off[u] + u
  int* n_feat;                        // [n_utt]
};

// K6 (level 11): cumulative 264-dim utterance distributions, one row per stored segment
struct FaUtteranceParams {
  const long long* frame_off;
  int n_utt;
  int utt_begin, utt_count;
  const fa_segment* segs; const int* n_segs;
  const fa_syllable* syls;
  const float* formants;
  const FaEpoch* epochs;              // see FaFeatureParams
  const long long* row_base;          // [n_utt + 1] first 264-row of every utterance in `rows` (capacity = difference)
  double* rows;
  int* n_feat;                        // [n_utt] rows written
  int* overflow;                      // [n_utt]
};

struct FaGatherArgs {
  const long long* frame_off;
  int n_utt;
  const FaEpoch* epochs;              // K3 stream mode: formant / energy rows are gathered segment by segment from the
                                      // epochs' frame ranges, several CTAs per utterance (row_slices); nullptr: contiguous
  int row_slices;
  int feat_width;                     // doubles per feature row: 53 (levels 5, 13), 23 (level 12) or 264 (level 11)
  int l3_mult;                        // level 3: maxp (the track headers in `syls` and the fa_track_point rows in `formants`
                                      // sit at base frame_off[u] * maxp); else 0
  const long long* feat_base;         // level 11: first row of every utterance in `features`; nullptr: frame_off[u] + u
  const int *n_segs, *n_rows, *n_syls, *n_feat;
  long long* off;  // [4][n_utt + 1] exclusive prefixes: segs, rows, syls, feat
  const fa_segment* segs; const fa_syllable* syls; const float* formants; const float* energy; const double* features;
  fa_segment* d_segs; fa_syllable* d_syls; float* d_formants; float* d_energy; double* d_features;
};

cudaError_t fa_launch_pcm_i16(const int16_t* src, float* dst, long long n, cudaStream_t s, int* launches);
// mid (optional): recorded between the frame-parallel |X|/N kernel and the smoothing / dB / band kernel
cudaError_t fa_launch_spectrum(const FaSpectrumParams& p, cudaStream_t s, int* launches, cudaEvent_t mid = nullptr);
cudaError_t fa_launch_peaks(const FaPeaksParams& p, cudaStream_t s, int* launches);
cudaError_t fa_launch_segment(const FaSegmentParams& p, cudaStream_t s, int* launches);
cudaError_t fa_launch_features(const FaFeatureParams& p, cudaStream_t s, int* launches);
int fa_mlp_run_device(fa_mlp* m, const double* d_rows, int n_rows, float* probs_host, cudaStream_t s);
int fa_mlp_in_dim(const fa_mlp* m);
int fa_mlp_device(const fa_mlp* m);
int fa_mlp_out_dim(const fa_mlp* m);
cudaError_t fa_launch_utterance(const FaUtteranceParams& p, cudaStream_t s, int* launches);
cudaError_t fa_launch_curves(const FaCurveParams& p, cudaStream_t s, int* launches);
cudaError_t fa_launch_prefix(const FaGatherArgs& a, cudaStream_t s, int* launches);
cudaError_t fa_launch_gather(const FaGatherArgs& a, cudaStream_t s, int* launches);
