// fa_capi.cu -- the C-ABI of libfa_b200.so (include/fa_b200.h): handles, batches, HBM layout, launches.
//
// HBM layout of one batch (all sizes derived from the submitted utterances; F = total frames):
//   pcm        float32 [sum of 4-aligned utterance lengths + pad]     read once by K1
//   spec_db    float32 [F][fft_size/2]         (only when the spectrum is wanted)      written once by K1
//   frames     uint32  [F][bands]              K1 -> K2, K3
//   cand/ncand/gsum  uint32 [F][maxp], int32 [F], float64 [F]       K2 -> K3
//   track table / point pool / row scratch     K3 workspace, per utterance, sized from its frame count
//   segs / syls / formants[F][9] / energy[F][3] / features          K3, K4 outputs, per-utterance regions
//   dense segs / syls / formants / energy / features + offsets      K5 gather -> one D2H copy each
// There is no CPU fallback: every entry point that computes needs the device.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <unordered_map>
#include <vector>

#include "fa_internal.cuh"
#include "fa_jsmath.h"
#include "fa_tables.h"

namespace {

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  cudaError_t reserve(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    size_t want = bytes + bytes / 8 + 256;
    cudaError_t e = cudaMalloc(&p, want);
    if (e != cudaSuccess) { e = cudaMalloc(&p, bytes); want = bytes; }
    if (e == cudaSuccess) cap = want;
    return e;
  }
  // as reserve(), and a NEW allocation is cleared once: for tables whose unused slots are loaded speculatively (K3 prefetches
  // candidate slot `lane` of the next frame before it knows the frame's count; the value is masked out, but the load would
  // read never-written memory -- compute-sanitizer initcheck)
  cudaError_t reserve_zeroed(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    cudaError_t e = reserve(bytes);
    if (e != cudaSuccess) return e;
    e = cudaMemset(p, 0, cap);
    if (e != cudaSuccess) return e;
    return cudaStreamSynchronize(cudaStreamLegacy);
  }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
  template <typename T> T* as() const { return reinterpret_cast<T*>(p); }
};

struct HostBuf {  // pinned
  void* p = nullptr;
  size_t cap = 0;
  cudaError_t reserve(size_t bytes, size_t keep = 0) {
    if (bytes <= cap) return cudaSuccess;
    size_t want = std::max(bytes, cap * 2);
    void* q = nullptr;
    cudaError_t e = cudaHostAlloc(&q, want, cudaHostAllocDefault);
    if (e != cudaSuccess) { want = bytes; e = cudaHostAlloc(&q, want, cudaHostAllocDefault); }
    if (e != cudaSuccess) return e;
    if (p && keep) memcpy(q, p, keep);
    if (p) cudaFreeHost(p);
    p = q;
    cap = want;
    return cudaSuccess;
  }
  void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
  template <typename T> T* as() const { return reinterpret_cast<T*>(p); }
};

struct Utt {
  int64_t id;
  int region;        // 0 = the handle's pinned staging buffer, > 0 = a caller-owned buffer (zero copy)
  long long off;     // first sample inside its region
  long long n;       // samples
  long long row0;    // first frame row
  int frames;
};

// A contiguous run of PCM on the host that maps to a contiguous run in d_pcm.
struct Region {
  const float* host;   // nullptr for region 0 (resolved at upload: the staging buffer may move while it grows)
  long long n;         // floats
  long long dev_off;   // first float in d_pcm (multiple of 4)
  const int16_t* host16 = nullptr;  // caller-owned int16 PCM (zero copy): crosses PCIe as int16, converted on the device
};

struct SubBatch { int u0, u1; long long r0, r1; };

constexpr int kMaxSub = 16;

}  // namespace

struct fa_handle {
  fa_config cfg;
  int device = 0;
  cudaStream_t own_stream = nullptr, stream = nullptr;
  std::string err;
  int sample_rate = 0, hop = 0, B = 0, N = 0, M = 0, logM = 0, maxp = 0;
  bool tables_ready = false;
  int tables_sr = 0;
  std::vector<Utt> utts;
  std::vector<Region> regions;
  std::vector<long long> abs_off;  // device offset of every utterance (filled by prepare)
  std::unordered_map<int64_t, int> index;
  long long staged = 0;        // floats used in h_pcm
  long long dev_floats = 0;    // floats of d_pcm in use
  int pipeline = 0;            // sub-batches: 0 = auto, 1 = serial
  void* spec_sink = nullptr;   // caller-owned destination of the spectrum rows (filled during fa_run), element type = spectrum_format
  size_t spec_sink_rows = 0;
  cudaStream_t sub_stream[kMaxSub] = {};
  cudaStream_t sub_hi[kMaxSub] = {};    // high-priority streams for the latency-bound segment scan + features of a sub-batch
  cudaEvent_t sub_done[kMaxSub] = {}, sub_mid[kMaxSub] = {}, sub_hi_done[kMaxSub] = {};
  cudaEvent_t spec_done[kMaxSub] = {}, copy_done[kMaxSub] = {};
  cudaStream_t own_copy_stream = nullptr, copy_stream = nullptr;
  // FA_TRACE=1: CUDA-event time stamps of every sub-batch (kernels start / spectrum done / D2H start / D2H end) against a
  // process-wide base event, printed by fa_sync (profiles/e2e_timeline)
  int prio_hi = 0, n_sub_streams = 0;
  bool trace = false;
  int trace_seq = 0;
  cudaEvent_t tr_ev[kMaxSub][4] = {};
  cudaEvent_t tr_k[kMaxSub][5] = {};   // resident runs: sub-batch start, after spectrum / peaks / segment / features  // spectrum-sink D2H, in sub-batch order (fa_set_d2h_stream)
  bool k3_priority = false;  // FA_K3_PRIO=1: measured slower on C2 (profiles/r1_sweep_overlap.txt), kept as a knob
  cudaEvent_t fork_ev = nullptr;
  bool prepared = false;
  long long total_frames = 0;
  HostBuf h_pcm, h_meta, h_counts, h_off, h_segs, h_syls, h_formants, h_energy, h_features;
  DevBuf d_pcm16;   // int16 PCM of caller regions, same element index as d_pcm
  DevBuf d_pcm, d_meta, d_spec, d_frames, d_cand, d_ncand, d_gsum, d_counter;
  DevBuf d_win, d_tw, d_tws, d_ws, d_bmi, d_bmw, d_emph;
  DevBuf d_spill, d_trkbase, d_trk_i, d_trk_d, d_trk_slot, d_pt_i, d_pt_e, d_rows, d_rowlist;
  DevBuf d_segs, d_syls, d_formants, d_energy, d_features, d_counts, d_off;
  // K1b stream mode: chunk work list (utt[], idx[], base[n+1]), speculated entry / true exit states, separate dB rows, fix-up count
  DevBuf d_chunks, d_state, d_specdb, d_fix;
  DevBuf d_specq;   // spectrum rows as uint8 (getByteFrequencyData) or half: [F][M] elements
  int chunk_frames = 0, warm_frames = 0;
  long long total_chunks = 0;
  std::vector<long long> chunk_base;   // host copy of base[]
  int fixups[3] = {-1, -1, -1};         // chunks recomputed in the last run by K1b / K3a, utterances redone by the general K3 (fetched lazily)
  // K3a stream mode: chunk work list, speculated entry / exit control states, T / k record of the gate's tests
  DevBuf d_cchunks, d_cstate, d_frT, d_frk, d_frthr;
  int ctl_chunk = 0, ctl_warm = 0;
  long long total_cchunks = 0;
  std::vector<long long> cchunk_base;
  float* spec_rows() const { return (chunk_frames > 0 && want_spec) ? d_specdb.as<float>() : d_spec.as<float>(); }
  // the rows the caller gets: float32 dB (in d_spec / d_specdb) or the uint8 / half rows of d_specq
  int spec_fmt() const { return cfg.spectrum_format; }
  size_t spec_elem() const { return spec_fmt() == FA_SPECTRUM_U8 ? 1 : spec_fmt() == FA_SPECTRUM_F16 ? 2 : 4; }
  const char* spec_out() const { return spec_fmt() == FA_SPECTRUM_F32 ? (const char*)spec_rows() : d_specq.as<char>(); }
  DevBuf d_frctl, d_frv, d_epochs, d_work, d_k3q;   // K3 mode 1: per-frame control record, epoch table, work list, queue counters
  int k3_cfg = -1;       // FA_K3_MODE: 0 = serial one-warp-per-utterance kernel, 1 = control scan + epoch-parallel tracking,
                         // unset = automatic (prepare): long utterances / streams take mode 1, short ones mode 0
  int k3_mode = 0;
  int k3_workers = 0;    // warps of the epoch-tracking grid
  int k3_impl = 2;       // FA_K3_IMPL: 2 = accumulate_fm2 kernel + redo launch (default), 1 = the general kernel alone
  int k3_warps = 0, k3_regs = 0, k3_finalize_smem = 1;   // FA_K3_WARPS, FA_K3_REGS, FA_K3_FINALIZE_HBM
  // K3 writes an epoch table + work list, and its rows sit at the epochs' first frames: mode 1, and the utterance-mode scan
  // whose finalisations run in their own launch (fa_segfin_kernel; not level 3, which finalises in the scan)
  bool k3_epochs() const { return k3_mode == 1 || (k3_impl == 2 && cfg.output_level != FA_LEVEL_SEGMENTS); }
  bool debug_sync = false;  // FA_DEBUG_SYNC
  int k1a_variant = 0;      // FA_K1A_VARIANT (see fa_launch_spectrum)
  int k1_fused = 0;         // FA_K1_FUSED=1: the fused K1 kernel (fft_size 2048, utterance mode) instead of K1a + K1b.  Measured
                            // slower on B200 (C2: 0.99 vs 0.94 ms with dB rows, 0.93 vs 0.86 ms without; the stage is FP32-issue
                            // bound and the fused kernel's barriers idle issue slots), so it is a knob: it moves 1.19 instead of
                            // 2.79 GB through HBM and needs no 4 KB-per-frame magnitude buffer when no dB rows are wanted
  bool use_fused() const { return k1_fused != 0 && N == 2048 && chunk_frames <= 0 && !frames_mode; }
  DevBuf g_segs, g_syls, g_formants, g_energy, g_features;
  DevBuf d_curve_work, d_curve_status, d_curve_list, d_curve_count;   // level 12 (K8)
  DevBuf d_pt_amp;                       // level 3: amplitudes of the pool points
  int no_truncate = 0;                   // fa_set_truncate(h, 0): prefixes of running streams
  size_t row_bytes() const { return cfg.output_level == FA_LEVEL_SEGMENTS ? sizeof(fa_track_point) : 9 * sizeof(float); }
  int n_weights = 0;
  long long track_total = 0, urow_total = 0;
  int feat_width() const {
    return cfg.output_level == FA_LEVEL_UTTERANCE ? FA_N_UTT_FEATURES : cfg.output_level == FA_LEVEL_SYL_CURVES ? FA_N_CURVE_FEATURES : FA_N_FEATURES;
  }
  bool uploaded = false, ran = false, downloaded = false, want_spec = false, from_host = false;
  bool frames_mode = false;    // the batch was submitted as uint32 frames (fa_submit_frames): the spectrum stage is skipped
  HostBuf h_frames;            // pinned staging of submitted frames, row order
  long long tot[4] = {0, 0, 0, 0};  // segs, rows, syls, feat
  bool have_table[5] = {false, false, false, false, false};   // dense tables fetched so far: segs, formants, energy, syls, features
  cudaEvent_t ev[8] = {};
  float stage_ms[5] = {0, 0, 0, 0, 0};
  float fft_ms = 0;   // first part of stage_ms[0]: the frame-parallel |X|/N kernel (serial mode)
  int launches = 0;
};

namespace {

int fail(fa_handle* h, int code, const char* what, cudaError_t e = cudaSuccess) {
  if (h) {
    h->err = what;
    if (e != cudaSuccess) { h->err += ": "; h->err += cudaGetErrorString(e); }
  }
  return code;
}

#define FA_CUDA(call)                                                        \
  do {                                                                       \
    cudaError_t e__ = (call);                                                \
    if (e__ != cudaSuccess) return fail(h, e__ == cudaErrorMemoryAllocation ? FA_ERR_OUT_OF_MEMORY : FA_ERR_CUDA, #call, e__); \
  } while (0)

bool level_supported(int lvl) {
  return lvl == FA_LEVEL_BARS || lvl == FA_LEVEL_SPECTRUM || lvl == FA_LEVEL_SEGMENTS || lvl == FA_LEVEL_FORMANTS || lvl == FA_LEVEL_SEG_FEATURES ||
         lvl == FA_LEVEL_SYL_FORMANTS || lvl == FA_LEVEL_UTTERANCE || lvl == FA_LEVEL_SYL_CURVES || lvl == FA_LEVEL_SYL_FEATURES;
}

int validate(const fa_config* c, std::string* why) {
  if (!fa_tab_valid_fft(c->fft_size)) { *why = "fft_size must be a power of two in [256, 16384]"; return FA_ERR_UNSUPPORTED; }
  if (!level_supported(c->output_level)) { *why = "output_level not supported (levels 1, 2, 3, 4, 5, 10, 11, 12, 13)"; return FA_ERR_UNSUPPORTED; }
  if (c->spec_type < 1 || c->spec_type > 3) { *why = "Invalid reset_nodes config"; return FA_ERR_INVALID_ARG; }
  const int B = fa_tab_bands(c);
  if (B < 8 || B > FA_MAX_BANDS) { *why = "Invalid spec_bands"; return FA_ERR_INVALID_ARG; }
  if (!(c->window_step_ms > 0) || !(c->f_max > c->f_min) || !(c->f_min >= 0)) { *why = "Invalid reset_nodes config"; return FA_ERR_INVALID_ARG; }
  if (c->spectrum_format < FA_SPECTRUM_F32 || c->spectrum_format > FA_SPECTRUM_F16) { *why = "spectrum_format must be FA_SPECTRUM_F32, _U8 or _F16"; return FA_ERR_INVALID_ARG; }
  if (c->spectrum_format == FA_SPECTRUM_U8 && !(c->max_db > c->min_db)) { *why = "maxDecibels must exceed minDecibels"; return FA_ERR_INVALID_ARG; }
  if (!(c->smoothing >= 0.0 && c->smoothing <= 1.0)) { *why = "smoothingTimeConstant must be in [0, 1]"; return FA_ERR_INVALID_ARG; }
  return FA_OK;
}

int build_tables(fa_handle* h, int sr) {
  const fa_config& c = h->cfg;
  const int N = c.fft_size, M = N / 2;
  h->N = N; h->M = M; h->logM = fa_tab_log2(M); h->B = fa_tab_bands(&c);
  h->hop = fa_tab_hop(sr, c.window_step_ms);
  h->maxp = h->B / 2 + 4;
  std::vector<float> win(N), tw(M), ws(2 * M), tws(2 * (size_t)(M - 1)), emph(h->B);
  fa_tab_window(N, win.data());
  fa_tab_fft_twiddles(M, tw.data());
  fa_tab_split_twiddles(M, ws.data());
  for (int s = 1; s <= h->logM; s++) {
    const int half = 1 << (s - 1), stride = M >> s, off = half - 1;
    for (int j = 0; j < half; j++) {
      tws[2 * (size_t)(off + j)] = tw[2 * (size_t)(j * stride)];
      tws[2 * (size_t)(off + j) + 1] = tw[2 * (size_t)(j * stride) + 1];
    }
  }
  fa_bandmat bm;
  if (fa_tab_bandmat(&c, sr, &bm) < 0) return fail(h, FA_ERR_OUT_OF_MEMORY, "band matrix");
  for (int m = 0; m < h->B; m++) emph[m] = (float)((double)m * c.high_f_emph);
  h->n_weights = bm.n_weights;
  std::vector<int> bmi(3 * (size_t)h->B + 1);
  for (int m = 0; m < h->B; m++) { bmi[m] = bm.k0[m]; bmi[h->B + m] = bm.cnt[m]; bmi[2 * h->B + m] = bm.off[m]; }
  bmi[3 * (size_t)h->B] = bm.off[h->B];
  cudaStream_t s = h->stream;
  int rc = FA_OK;
  do {
#define FA_UP(buf, vec)                                                                                   \
  {                                                                                                       \
    cudaError_t e = buf.reserve(std::max<size_t>(16, vec.size() * sizeof(vec[0])));                      \
    if (e == cudaSuccess && !vec.empty())                                                                 \
      e = cudaMemcpyAsync(buf.p, vec.data(), vec.size() * sizeof(vec[0]), cudaMemcpyHostToDevice, s);     \
    if (e != cudaSuccess) { rc = fail(h, FA_ERR_CUDA, "table upload", e); break; }                        \
  }
    FA_UP(h->d_win, win);
    FA_UP(h->d_tw, tw);
    FA_UP(h->d_tws, tws);
    FA_UP(h->d_ws, ws);
    FA_UP(h->d_bmi, bmi);
    FA_UP(h->d_emph, emph);
    {
      std::vector<float> w(bm.w, bm.w + std::max(1, bm.n_weights));
      FA_UP(h->d_bmw, w);
    }
#undef FA_UP
    cudaError_t e = cudaStreamSynchronize(s);  // the vectors above die at scope exit
    if (e != cudaSuccess) rc = fail(h, FA_ERR_CUDA, "table upload sync", e);
  } while (0);
  fa_tab_bandmat_free(&bm);
  if (rc == FA_OK) { h->tables_ready = true; h->tables_sr = sr; }
  return rc;
}

Utt* find_utt(fa_handle* h, int64_t id) {
  auto it = h->index.find(id);
  return it == h->index.end() ? nullptr : &h->utts[it->second];
}

}  // namespace

extern "C" {

void fa_config_default(fa_config* c) {
  memset(c, 0, sizeof(*c));
  c->spec_type = 1; c->output_level = 4; c->plot_len = 200; c->n_fft_bins = 256; c->n_mel_bins = 128;
  c->auto_noise_gate = 1; c->f_min = 50; c->f_max = 4000; c->window_width_ms = 25; c->window_step_ms = 25;
  c->pause_length_ms = 200; c->min_seg_length_ms = 50; c->voiced_max_db = 100; c->voiced_min_db = 10;
  c->pre_norm_gain = 1000; c->high_f_emph = 0; c->fft_size = 2048; c->clamp_db = 1; c->want_spectrum = 0;
  c->smoothing = 0.8; c->min_db = -100; c->max_db = -30; c->mag_scale = 0;
}

int fa_abi_version(void) { return FA_ABI_VERSION; }

const char* fa_status_string(int s) {
  switch (s) {
    case FA_OK: return "ok";
    case FA_ERR_INVALID_ARG: return "invalid argument";
    case FA_ERR_NO_DEVICE: return "no usable sm_100 CUDA device (there is no CPU fallback)";
    case FA_ERR_CUDA: return "CUDA error";
    case FA_ERR_NOT_RUN: return "results requested before fa_run/fa_sync";
    case FA_ERR_UNKNOWN_UTT: return "unknown utterance id";
    case FA_ERR_CAPACITY: return "capacity exceeded";
    case FA_ERR_OUT_OF_MEMORY: return "out of memory";
    case FA_ERR_BUSY: return "Error: Already playing";
    case FA_ERR_UNSUPPORTED: return "unsupported configuration";
    default: return "unknown status";
  }
}

int fa_hop_samples(const fa_config* c, int sr) { return fa_tab_hop(sr, c->window_step_ms); }
int fa_frames_for(const fa_config* c, int sr, size_t n) { return (int)(n / (size_t)fa_tab_hop(sr, c->window_step_ms)); }
int fa_spec_bands(const fa_config* c) { return fa_tab_bands(c); }

int fa_create(const fa_config* cfg, int device, fa_handle** out) {
  if (!cfg || !out) return FA_ERR_INVALID_ARG;
  *out = nullptr;
  std::string why;
  const int v = validate(cfg, &why);
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0 || device < 0 || device >= ndev) return FA_ERR_NO_DEVICE;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess || prop.major != 10) return FA_ERR_NO_DEVICE;
  if (v != FA_OK) return v;
  fa_handle* h = new fa_handle();
  h->cfg = *cfg;
  h->device = device;
  if (cudaSetDevice(device) != cudaSuccess || cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking) != cudaSuccess) {
    delete h;
    return FA_ERR_CUDA;
  }
  h->stream = h->own_stream;
  for (auto& e : h->ev) cudaEventCreate(&e);
  int prio_lo = 0, prio_hi = 0;
  cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);  // numerically lowest = greatest priority
  if (const char* ev = getenv("FA_K3_PRIO")) h->k3_priority = atoi(ev) != 0;
  if (const char* ev = getenv("FA_TRACE")) h->trace = atoi(ev) != 0;
  if (const char* ev = getenv("FA_K3_MODE")) h->k3_cfg = atoi(ev) != 0;
  h->k3_workers = prop.multiProcessorCount * 14;   // 7 CTAs x 2 warps per SM (shared memory bound)
  if (const char* ev = getenv("FA_K3_WORKERS")) { const int v = atoi(ev); if (v >= 32 && v <= 1 << 16) h->k3_workers = v; }
  // every environment knob is read here, once per handle -- nothing on the launch path calls getenv
  if (const char* ev = getenv("FA_K3_IMPL")) { const int v = atoi(ev); h->k3_impl = v == 1 ? 1 : v == 3 ? 3 : 2; }
  if (const char* ev = getenv("FA_K3_WARPS")) { const int v = atoi(ev); if (v >= 1 && v <= 4) h->k3_warps = v; }
  if (const char* ev = getenv("FA_K3_REGS")) h->k3_regs = atoi(ev);
  if (getenv("FA_K3_FINALIZE_HBM")) h->k3_finalize_smem = 0;
  if (getenv("FA_DEBUG_SYNC")) h->debug_sync = true;
  if (const char* ev = getenv("FA_K1_FUSED")) h->k1_fused = atoi(ev) != 0;
  if (const char* ev = getenv("FA_K1A_VARIANT")) h->k1a_variant = atoi(ev);

  // Streams are created on first use (ensure_sub_streams): the device has at most 32 hardware work queues
  // (CUDA_DEVICE_MAX_CONNECTIONS, default 8) and streams beyond that alias onto the same queue, where a stream that waits
  // for a long D2H falsely blocks its queue mates -- measured: with 34 streams per handle two handles never overlapped.
  h->prio_hi = prio_hi;
  cudaEventCreateWithFlags(&h->fork_ev, cudaEventDisableTiming);
  h->want_spec = cfg->want_spectrum || cfg->output_level <= 2;
  h->regions.push_back(Region{nullptr, 0, 0});
  *out = h;
  return FA_OK;
}

int fa_destroy(fa_handle* h) {
  if (!h) return FA_OK;
  cudaSetDevice(h->device);
  cudaStreamSynchronize(h->stream);
  for (int i = 0; i < kMaxSub; i++) if (h->sub_stream[i]) cudaStreamSynchronize(h->sub_stream[i]);
  for (int i = 0; i < kMaxSub; i++) if (h->sub_hi[i]) cudaStreamSynchronize(h->sub_hi[i]);
  for (DevBuf* b : {&h->d_pcm16, &h->d_pcm, &h->d_meta, &h->d_spec, &h->d_frames, &h->d_cand, &h->d_ncand, &h->d_gsum, &h->d_counter,
                    &h->d_win, &h->d_tw, &h->d_tws, &h->d_ws, &h->d_bmi, &h->d_bmw, &h->d_emph, &h->d_spill, &h->d_trkbase, &h->d_trk_i,
                    &h->d_trk_d, &h->d_trk_slot, &h->d_pt_i, &h->d_pt_e, &h->d_rows, &h->d_rowlist, &h->d_segs, &h->d_syls,
                    &h->d_formants, &h->d_energy, &h->d_features, &h->d_counts, &h->d_off, &h->g_segs, &h->g_syls,
                    &h->g_formants, &h->g_energy, &h->g_features, &h->d_chunks, &h->d_state, &h->d_specdb, &h->d_specq, &h->d_fix, &h->d_cchunks, &h->d_cstate, &h->d_frT, &h->d_frk, &h->d_frthr, &h->d_frctl, &h->d_frv, &h->d_epochs, &h->d_work, &h->d_k3q, &h->d_curve_work, &h->d_curve_status, &h->d_curve_list, &h->d_curve_count, &h->d_pt_amp})
    b->release();
  for (HostBuf* b : {&h->h_pcm, &h->h_frames, &h->h_meta, &h->h_counts, &h->h_off, &h->h_segs, &h->h_syls, &h->h_formants, &h->h_energy,
                     &h->h_features})
    b->release();
  for (auto& e : h->ev) if (e) cudaEventDestroy(e);
  for (int i = 0; i < kMaxSub; i++) {
    if (h->sub_done[i]) cudaEventDestroy(h->sub_done[i]);
    if (h->sub_mid[i]) cudaEventDestroy(h->sub_mid[i]);
    if (h->sub_hi_done[i]) cudaEventDestroy(h->sub_hi_done[i]);
    if (h->spec_done[i]) cudaEventDestroy(h->spec_done[i]);
    if (h->copy_done[i]) cudaEventDestroy(h->copy_done[i]);
    for (int k = 0; k < 4; k++) if (h->tr_ev[i][k]) cudaEventDestroy(h->tr_ev[i][k]);
    if (h->sub_stream[i]) cudaStreamDestroy(h->sub_stream[i]);
    if (h->sub_hi[i]) cudaStreamDestroy(h->sub_hi[i]);
  }
  if (h->fork_ev) cudaEventDestroy(h->fork_ev);
  if (h->own_copy_stream) { cudaStreamSynchronize(h->own_copy_stream); cudaStreamDestroy(h->own_copy_stream); }
  if (h->own_stream) cudaStreamDestroy(h->own_stream);
  delete h;
  return FA_OK;
}

const char* fa_last_error(const fa_handle* h) { return h ? h->err.c_str() : "null handle"; }

void* fa_host_alloc(size_t bytes, int write_combined) {
  void* p = nullptr;
  const unsigned flags = cudaHostAllocPortable | (write_combined ? cudaHostAllocWriteCombined : 0u);
  if (cudaHostAlloc(&p, bytes ? bytes : 1, flags) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  return p;
}
void fa_host_free(void* p) { if (p) cudaFreeHost(p); }

int fa_pcie_probe(int device, void* host, size_t bytes, int reps, int direction, float* ms_per_copy) {
  if (!host || !bytes || reps <= 0 || !ms_per_copy || direction < 0 || direction > 1) return FA_ERR_INVALID_ARG;
  if (cudaSetDevice(device) != cudaSuccess) return FA_ERR_NO_DEVICE;
  void* d = nullptr;
  cudaStream_t s = nullptr;
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  int rc = FA_OK;
  if (cudaMalloc(&d, bytes) != cudaSuccess) { cudaGetLastError(); return FA_ERR_OUT_OF_MEMORY; }
  if (cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking) != cudaSuccess || cudaEventCreate(&e0) != cudaSuccess ||
      cudaEventCreate(&e1) != cudaSuccess) rc = FA_ERR_CUDA;
  if (rc == FA_OK) {
    const cudaMemcpyKind kind = direction == 0 ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToHost;
    cudaMemcpyAsync(direction == 0 ? d : host, direction == 0 ? host : d, bytes, kind, s);   // warm-up
    cudaEventRecord(e0, s);
    for (int i = 0; i < reps; i++) cudaMemcpyAsync(direction == 0 ? d : host, direction == 0 ? host : d, bytes, kind, s);
    cudaEventRecord(e1, s);
    float ms = 0.f;
    if (cudaStreamSynchronize(s) != cudaSuccess || cudaEventElapsedTime(&ms, e0, e1) != cudaSuccess) rc = FA_ERR_CUDA;
    *ms_per_copy = ms / (float)reps;
  }
  if (e0) cudaEventDestroy(e0);
  if (e1) cudaEventDestroy(e1);
  if (s) cudaStreamDestroy(s);
  cudaFree(d);
  if (rc != FA_OK) cudaGetLastError();
  return rc;
}

int fa_get_config(const fa_handle* h, fa_config* out) {
  if (!h || !out) return FA_ERR_INVALID_ARG;
  *out = h->cfg;
  return FA_OK;
}

int fa_set_stream(fa_handle* h, void* s) {
  if (!h) return FA_ERR_INVALID_ARG;
  cudaSetDevice(h->device);
  cudaStreamSynchronize(h->stream);
  h->stream = s ? reinterpret_cast<cudaStream_t>(s) : h->own_stream;
  return FA_OK;
}

int fa_set_d2h_stream(fa_handle* h, void* s) {
  if (!h) return FA_ERR_INVALID_ARG;
  cudaSetDevice(h->device);
  if (h->copy_stream) cudaStreamSynchronize(h->copy_stream);
  h->copy_stream = s ? reinterpret_cast<cudaStream_t>(s) : h->own_copy_stream;
  return FA_OK;
}

int fa_set_pipeline(fa_handle* h, int n_sub) {
  if (!h || n_sub < 0 || n_sub > kMaxSub) return FA_ERR_INVALID_ARG;
  h->pipeline = n_sub;
  return FA_OK;
}

int fa_set_spectrum_sink_raw(fa_handle* h, void* dst, size_t cap_rows) {
  if (!h) return FA_ERR_INVALID_ARG;
  if (dst && !h->want_spec) return fail(h, FA_ERR_INVALID_ARG, "spectrum not materialised (set want_spectrum or output_level <= 2)");
  h->spec_sink = dst;
  h->spec_sink_rows = dst ? cap_rows : 0;
  return FA_OK;
}

int fa_set_spectrum_sink(fa_handle* h, float* dst, size_t cap_rows) {
  if (!h) return FA_ERR_INVALID_ARG;
  if (dst && h->spec_fmt() != FA_SPECTRUM_F32) return fail(h, FA_ERR_INVALID_ARG, "spectrum_format is not float32: use fa_set_spectrum_sink_raw");
  return fa_set_spectrum_sink_raw(h, dst, cap_rows);
}

int fa_reset(fa_handle* h) {
  if (!h) return FA_ERR_INVALID_ARG;
  cudaSetDevice(h->device);
  cudaStreamSynchronize(h->stream);
  h->utts.clear();
  h->index.clear();
  h->regions.clear();
  h->regions.push_back(Region{nullptr, 0, 0});
  h->staged = 0;
  h->total_frames = 0;
  h->uploaded = h->ran = h->downloaded = h->prepared = false;
  h->frames_mode = false;
  return FA_OK;
}

static int add_utt(fa_handle* h, int64_t utt_id, int region, long long off, size_t n, int sr) {
  if (utt_id < 0) return fail(h, FA_ERR_INVALID_ARG, "utterance ids must be >= 0 (FA_ALL_UTTS = -1 names the whole batch)");
  if (h->index.count(utt_id)) return fail(h, FA_ERR_INVALID_ARG, "duplicate utterance id");
  Utt u;
  u.id = utt_id; u.region = region; u.off = off; u.n = (long long)n;
  u.frames = (int)(n / (size_t)fa_tab_hop(sr, h->cfg.window_step_ms));
  u.row0 = h->total_frames;
  h->index[utt_id] = (int)h->utts.size();
  h->utts.push_back(u);
  h->total_frames += u.frames;
  return (int)h->utts.size() - 1;
}

static int submit_check(fa_handle* h, int sr) {
  if (!h || sr <= 0) return fail(h, FA_ERR_INVALID_ARG, "Invalid audio source");
  cudaSetDevice(h->device);
  if (h->uploaded || h->ran) return fail(h, FA_ERR_BUSY, "Error: Already playing");
  if (h->frames_mode) return fail(h, FA_ERR_INVALID_ARG, "a batch holds either PCM or frames, not both");
  if (h->utts.empty()) h->sample_rate = sr;
  else if (sr != h->sample_rate) return fail(h, FA_ERR_INVALID_ARG, "all utterances of a batch must share the sample rate");
  return FA_OK;
}

static int submit_common(fa_handle* h, int64_t utt_id, size_t n, int sr, float** dst) {
  int rc = submit_check(h, sr);
  if (rc != FA_OK) return rc;
  if (utt_id < 0) return fail(h, FA_ERR_INVALID_ARG, "utterance ids must be >= 0 (FA_ALL_UTTS = -1 names the whole batch)");
  if (h->index.count(utt_id)) return fail(h, FA_ERR_INVALID_ARG, "duplicate utterance id");
  const long long off = h->staged;
  const long long padded = ((long long)n + 3) & ~3ll;
  FA_CUDA(h->h_pcm.reserve((size_t)(off + padded + 16) * sizeof(float), (size_t)off * sizeof(float)));
  rc = add_utt(h, utt_id, 0, off, n, sr);
  if (rc < 0) return rc;
  h->staged = off + padded;
  *dst = h->h_pcm.as<float>() + off;
  for (long long i = (long long)n; i < padded; i++) (*dst)[i] = 0.f;
  return rc;
}

int fa_submit_pcm(fa_handle* h, int64_t utt_id, const float* pcm, size_t n, int sr) {
  if (!pcm && n) return fail(h, FA_ERR_INVALID_ARG, "Invalid audio source");
  float* dst = nullptr;
  const int rc = submit_common(h, utt_id, n, sr, &dst);
  if (rc < 0) return rc;
  if (n) memcpy(dst, pcm, n * sizeof(float));
  return rc;
}

int fa_submit_pcm_i16(fa_handle* h, int64_t utt_id, const int16_t* pcm, size_t n, int sr) {
  if (!pcm && n) return fail(h, FA_ERR_INVALID_ARG, "Invalid audio source");
  float* dst = nullptr;
  const int rc = submit_common(h, utt_id, n, sr, &dst);
  if (rc < 0) return rc;
  for (size_t i = 0; i < n; i++) dst[i] = (float)pcm[i] * (1.0f / 32768.0f);
  return rc;
}

int fa_submit_pcm_batch(fa_handle* h, int64_t first_utt_id, const float* pcm, const int64_t* offsets, int n_utt, int sr) {
  int rc = submit_check(h, sr);
  if (rc != FA_OK) return rc;
  if (!pcm || !offsets || n_utt <= 0) return fail(h, FA_ERR_INVALID_ARG, "Invalid audio source");
  for (int i = 0; i < n_utt; i++)
    if (offsets[i + 1] < offsets[i] || offsets[0] < 0) return fail(h, FA_ERR_INVALID_ARG, "offsets must be non-decreasing");
  if (first_utt_id < 0) return fail(h, FA_ERR_INVALID_ARG, "utterance ids must be >= 0 (FA_ALL_UTTS = -1 names the whole batch)");
  for (int i = 0; i < n_utt; i++)
    if (h->index.count(first_utt_id + i)) return fail(h, FA_ERR_INVALID_ARG, "duplicate utterance id");
  cudaPointerAttributes attr;
  const bool pinned = cudaPointerGetAttributes(&attr, pcm) == cudaSuccess && attr.type == cudaMemoryTypeHost;
  cudaGetLastError();  // an unregistered pointer is not an error for us
  const int first = (int)h->utts.size();
  if (pinned) {
    // zero copy: the H2D transfer reads the caller's buffer, which must stay valid until fa_sync
    Region r;
    r.host = pcm + offsets[0];
    r.n = offsets[n_utt] - offsets[0];
    r.dev_off = 0;
    h->regions.push_back(r);
    const int ri = (int)h->regions.size() - 1;
    for (int i = 0; i < n_utt; i++) {
      rc = add_utt(h, first_utt_id + i, ri, offsets[i] - offsets[0], (size_t)(offsets[i + 1] - offsets[i]), sr);
      if (rc < 0) return rc;
    }
  } else {
    for (int i = 0; i < n_utt; i++) {
      rc = fa_submit_pcm(h, first_utt_id + i, pcm + offsets[i], (size_t)(offsets[i + 1] - offsets[i]), sr);
      if (rc < 0) return rc;
    }
  }
  return first;
}

int fa_submit_pcm_i16_batch(fa_handle* h, int64_t first_utt_id, const int16_t* pcm, const int64_t* offsets, int n_utt, int sr) {
  int rc = submit_check(h, sr);
  if (rc != FA_OK) return rc;
  if (!pcm || !offsets || n_utt <= 0) return fail(h, FA_ERR_INVALID_ARG, "Invalid audio source");
  for (int i = 0; i < n_utt; i++)
    if (offsets[i + 1] < offsets[i] || offsets[0] < 0) return fail(h, FA_ERR_INVALID_ARG, "offsets must be non-decreasing");
  if (first_utt_id < 0) return fail(h, FA_ERR_INVALID_ARG, "utterance ids must be >= 0 (FA_ALL_UTTS = -1 names the whole batch)");
  for (int i = 0; i < n_utt; i++)
    if (h->index.count(first_utt_id + i)) return fail(h, FA_ERR_INVALID_ARG, "duplicate utterance id");
  cudaPointerAttributes attr;
  const bool pinned = cudaPointerGetAttributes(&attr, pcm) == cudaSuccess && attr.type == cudaMemoryTypeHost;
  cudaGetLastError();
  const int first = (int)h->utts.size();
  if (pinned) {
    Region r;
    r.host = nullptr;
    r.host16 = pcm + offsets[0];
    r.n = offsets[n_utt] - offsets[0];
    r.dev_off = 0;
    h->regions.push_back(r);
    const int ri = (int)h->regions.size() - 1;
    for (int i = 0; i < n_utt; i++) {
      rc = add_utt(h, first_utt_id + i, ri, offsets[i] - offsets[0], (size_t)(offsets[i + 1] - offsets[i]), sr);
      if (rc < 0) return rc;
    }
  } else {
    for (int i = 0; i < n_utt; i++) {
      rc = fa_submit_pcm_i16(h, first_utt_id + i, pcm + offsets[i], (size_t)(offsets[i + 1] - offsets[i]), sr);
      if (rc < 0) return rc;
    }
  }
  return first;
}

int fa_submit_frames(fa_handle* h, int64_t utt_id, const uint32_t* frames, size_t n_frames, int bands) {
  if (!h) return FA_ERR_INVALID_ARG;
  cudaSetDevice(h->device);
  if (h->uploaded || h->ran) return fail(h, FA_ERR_BUSY, "Error: Already playing");
  if (!h->frames_mode && !h->utts.empty()) return fail(h, FA_ERR_INVALID_ARG, "a batch holds either PCM or frames, not both");
  if (h->cfg.output_level < 3) return fail(h, FA_ERR_INVALID_ARG, "frames carry no spectrum: output_level must be >= 3");
  const int B = fa_tab_bands(&h->cfg);
  if (bands != B) return fail(h, FA_ERR_INVALID_ARG, "Error: bins num mismatch");   // spectrum_push's own check @B30392
  if (!frames && n_frames) return fail(h, FA_ERR_INVALID_ARG, "Invalid audio source");
  if (n_frames > (size_t)INT32_MAX) return fail(h, FA_ERR_CAPACITY, "too many frames");
  if (utt_id < 0) return fail(h, FA_ERR_INVALID_ARG, "utterance ids must be >= 0 (FA_ALL_UTTS = -1 names the whole batch)");
  if (h->index.count(utt_id)) return fail(h, FA_ERR_INVALID_ARG, "duplicate utterance id");
  if (h->sample_rate <= 0) h->sample_rate = 16000;   // only sizes the (unused) spectrum tables
  const size_t row = (size_t)B * sizeof(uint32_t);
  const size_t used = (size_t)h->total_frames * row;
  FA_CUDA(h->h_frames.reserve(used + n_frames * row + 64, used));
  if (n_frames) memcpy((char*)h->h_frames.p + used, frames, n_frames * row);
  Utt u;
  u.id = utt_id; u.region = 0; u.off = 0; u.n = 0; u.frames = (int)n_frames; u.row0 = h->total_frames;
  h->index[utt_id] = (int)h->utts.size();
  h->utts.push_back(u);
  h->total_frames += u.frames;
  h->frames_mode = true;
  return (int)h->utts.size() - 1;
}

// allocate everything a run needs and upload the small tables / metadata (not the PCM)
static int prepare(fa_handle* h) {
  if (h->utts.empty()) return fail(h, FA_ERR_INVALID_ARG, "Invalid audio source");
  if (!h->tables_ready || h->tables_sr != h->sample_rate) {
    const int rc = build_tables(h, h->sample_rate);
    if (rc != FA_OK) return rc;
  }
  const int n = (int)h->utts.size();
  const long long F = h->total_frames;
  cudaStream_t s = h->stream;
  // K3 mode: the split costs one extra (cheap) sequential pass per frame and pays off when an utterance holds many
  // segments -- measured on B200: C2 (200 frames, 1.75 segments per utterance) 1.18 ms serial vs 1.38 ms split, the
  // one-hour stream (144 000 frames, 541 segments) 641 ms serial vs 124 ms split
  h->k3_mode = h->k3_cfg >= 0 ? h->k3_cfg : (F / std::max(n, 1) >= 1000 ? 1 : 0);
  if (h->cfg.output_level == FA_LEVEL_SEGMENTS) h->k3_mode = 0;   // the raw-track export lives in the serial scan's finalisation
  // K1b stream mode for the same long utterances: chunks of 2048 frames, warm-up long enough for tau^W << 2^-24 plus a
  // margin for the last-ulp coalescence (FA_K1B_CHUNK=0 disables, FA_K1B_WARMUP overrides W -- the tests force W = 8 to
  // exercise the fix-up pass); tau close to 1 would need a warm-up as long as a chunk: one pass per utterance then
  {
    int ch = (F / std::max(n, 1) >= 1000 && !h->frames_mode) ? 2048 : 0;
    if (const char* ev = getenv("FA_K1B_CHUNK")) ch = atoi(ev);
    int warm = 0;
    if (ch > 0) {
      const double tau = h->cfg.smoothing;
      warm = tau <= 0.0 ? 8 : (int)ceil(40.0 * log(2.0) / -log(tau)) + 64;
      if (const char* ev = getenv("FA_K1B_WARMUP")) warm = atoi(ev);
      warm = std::max(8, (warm + 7) & ~7);
      ch = std::max(64, (ch + 7) & ~7);
      if (!(tau < 1.0) || warm > ch / 2) ch = 0;
    }
    h->chunk_frames = ch; h->warm_frames = ch ? warm : 0;
  }
  // K3a stream mode: chunks of 4096 frames scanned from a speculated state (warm-up 1024 frames: a few segments, so that both
  // the gate -- renewed by every frame louder than y -- and the segment state -- renewed by every finalisation -- have been
  // through a renewal); FA_K3_CHUNK=0 disables, FA_K3_WARM overrides (tests force a useless warm-up)
  {
    int ch = (h->k3_mode == 1 && F / std::max(n, 1) >= 1000) ? 4096 : 0;
    if (const char* ev = getenv("FA_K3_CHUNK")) ch = h->k3_mode == 1 ? atoi(ev) : 0;
    int warm = 1024;
    if (const char* ev = getenv("FA_K3_WARM")) warm = atoi(ev);
    h->ctl_chunk = ch > 0 ? std::max(16, ch) : 0;
    h->ctl_warm = std::max(0, warm);
  }
  // device layout of the PCM: [staging | caller buffers ...], each region 16-byte aligned
  long long dev = 0;
  h->regions[0].n = h->staged;
  for (auto& r : h->regions) {
    r.dev_off = dev;
    dev += (r.n + 3) & ~3ll;
  }
  h->dev_floats = dev;
  h->abs_off.resize(n);
  // meta: utt_off[n], utt_len[n], frame_off[n+1], track_base[n+1], urow_base[n+1]
  FA_CUDA(h->h_meta.reserve(sizeof(long long) * (5 * (size_t)n + 3)));
  long long* m = h->h_meta.as<long long>();
  long long tb = 0, ub = 0;
  // level 11: a stored segment spans > seg_min_frames voiced frames plus >= seg_breaker pause frames (none for the last one)
  const double brk = h->cfg.pause_length_ms > 2 * h->cfg.window_step_ms ? h->cfg.pause_length_ms / h->cfg.window_step_ms
                                                                         : 250 / h->cfg.window_step_ms;
  const long long seg_span = (long long)fa_js_parse_int(h->cfg.min_seg_length_ms / h->cfg.window_step_ms) + 1 + (long long)ceil(brk);
  for (int i = 0; i < n; i++) {
    const Utt& u = h->utts[i];
    h->abs_off[i] = h->regions[u.region].dev_off + u.off;
    m[i] = h->abs_off[i];
    m[n + i] = u.n;
    m[2 * n + i] = u.row0;
    m[3 * n + 1 + i] = tb;
    // track table: tracks <= points <= accepted peaks <= maxp per frame, so `maxp` entries per frame can never overflow
    // (mode 1 gives every epoch its own frame range of the table); the pages nobody touches cost nothing
    tb += (long long)u.frames * h->maxp + 64;
    m[4 * n + 2 + i] = ub;
    ub += u.frames / std::max<long long>(seg_span, 1) + 2;
  }
  m[2 * n + n] = F;
  m[3 * n + 1 + n] = tb;
  m[4 * n + 2 + n] = ub;
  h->track_total = tb;
  h->urow_total = ub;
  FA_CUDA(h->d_meta.reserve(sizeof(long long) * (5 * (size_t)n + 3)));
  FA_CUDA(cudaMemcpyAsync(h->d_meta.p, m, sizeof(long long) * (5 * (size_t)n + 3), cudaMemcpyHostToDevice, s));
  FA_CUDA(h->d_pcm.reserve((size_t)(dev + 16) * sizeof(float)));
  {
    bool any16 = false;
    for (const auto& r : h->regions) any16 = any16 || r.host16;
    if (any16) FA_CUDA(h->d_pcm16.reserve((size_t)(dev + 16) * sizeof(int16_t)));
  }
  const size_t Fz = (size_t)std::max<long long>(F, 1), nz = (size_t)n;
  // the K1a -> K1b magnitude rows, turned into dB rows in place; the fused kernel needs them only as dB output
  if (h->want_spec || !h->use_fused()) FA_CUDA(h->d_spec.reserve(Fz * h->M * sizeof(float)));
  if (h->want_spec && h->spec_fmt() != FA_SPECTRUM_F32) FA_CUDA(h->d_specq.reserve(Fz * h->M * h->spec_elem()));
  FA_CUDA(h->d_frames.reserve(Fz * h->B * sizeof(uint32_t)));
  FA_CUDA(h->d_counter.reserve(2 * kMaxSub * sizeof(int)));
  if (h->cfg.output_level >= 3) {
    FA_CUDA(h->d_cand.reserve_zeroed(Fz * h->maxp * sizeof(FaCand)));
    FA_CUDA(h->d_ncand.reserve(Fz * sizeof(int)));
    FA_CUDA(h->d_gsum.reserve(Fz * sizeof(double)));
    const size_t T = (size_t)std::max<long long>(tb, 1);
    FA_CUDA(h->d_trk_i.reserve(T * 3 * sizeof(int)));        // count, order, rank
    FA_CUDA(h->d_trk_d.reserve(T * 3 * sizeof(double)));     // sum_e, sum_eb, mean
    FA_CUDA(h->d_trk_slot.reserve(T));
    const size_t P = Fz * h->maxp;
    FA_CUDA(h->d_pt_i.reserve(P * 4 * sizeof(int)));         // track, ord, frame, binspan
    FA_CUDA(h->d_pt_e.reserve(P * sizeof(double)));
    FA_CUDA(h->d_rows.reserve((Fz + nz) * 2 * sizeof(int)));
    FA_CUDA(h->d_rowlist.reserve(P * sizeof(int)));
    FA_CUDA(h->d_spill.reserve(std::max<size_t>(nz, (size_t)h->k3_workers) * 6 * 128 * sizeof(unsigned long long)));
    if (h->k3_mode == 1) {
      FA_CUDA(h->d_frctl.reserve(Fz * sizeof(unsigned)));
      FA_CUDA(h->d_frv.reserve(Fz * sizeof(double)));
    }
    if (h->k3_epochs()) {
      FA_CUDA(h->d_epochs.reserve((Fz + nz) * sizeof(FaEpoch)));
      FA_CUDA(h->d_work.reserve((Fz + nz) * sizeof(int2)));
      FA_CUDA(h->d_k3q.reserve(2 * kMaxSub * sizeof(int)));
    }
    const bool l3 = h->cfg.output_level == FA_LEVEL_SEGMENTS;
    // level 3: the "syllable" table holds the fa_track headers and the "formant row" table the fa_track_point rows of the
    // ranked tracks, both with the capacity (and base) of the point pool
    static_assert(sizeof(fa_track) == sizeof(fa_syllable) && sizeof(fa_track_point) == 24, "level-3 tables reuse the row plumbing");
    FA_CUDA(h->d_segs.reserve((Fz + nz) * sizeof(fa_segment)));
    FA_CUDA(h->d_syls.reserve(l3 ? P * sizeof(fa_track) : (Fz + nz) * sizeof(fa_syllable)));
    FA_CUDA(h->d_formants.reserve(l3 ? P * sizeof(fa_track_point) : Fz * 9 * sizeof(float)));
    FA_CUDA(h->d_energy.reserve(Fz * 3 * sizeof(float)));
    if (l3) FA_CUDA(h->d_pt_amp.reserve(P * sizeof(int)));
    if (h->cfg.output_level == 5 || h->cfg.output_level == 13 || h->cfg.output_level == FA_LEVEL_SYL_CURVES)
      FA_CUDA(h->d_features.reserve((Fz + nz) * h->feat_width() * sizeof(double)));
    if (h->cfg.output_level == FA_LEVEL_SYL_CURVES) {
      FA_CUDA(h->d_curve_work.reserve(Fz * 34 * sizeof(double)));
      FA_CUDA(h->d_curve_status.reserve((Fz + nz) * 4 * sizeof(int)));
      FA_CUDA(h->d_curve_list.reserve((Fz + nz) * sizeof(int2)));
      FA_CUDA(h->d_curve_count.reserve(kMaxSub * sizeof(int)));
    }
    if (h->cfg.output_level == FA_LEVEL_UTTERANCE) {
      FA_CUDA(h->d_features.reserve((size_t)ub * FA_N_UTT_FEATURES * sizeof(double)));
      FA_CUDA(h->g_features.reserve((size_t)ub * FA_N_UTT_FEATURES * sizeof(double)));
    }
    FA_CUDA(h->d_counts.reserve(nz * 6 * sizeof(int)));      // n_segs, n_stored, n_rows, n_syls, n_feat, overflow
    FA_CUDA(h->d_off.reserve((nz + 1) * 4 * sizeof(long long)));
    FA_CUDA(h->g_segs.reserve((Fz + nz) * sizeof(fa_segment)));
    FA_CUDA(h->g_syls.reserve(l3 ? P * sizeof(fa_track) : (Fz + nz) * sizeof(fa_syllable)));
    FA_CUDA(h->g_formants.reserve(l3 ? P * sizeof(fa_track_point) : Fz * 9 * sizeof(float)));
    FA_CUDA(h->g_energy.reserve(Fz * 3 * sizeof(float)));
    if (h->cfg.output_level == 5 || h->cfg.output_level == 13 || h->cfg.output_level == FA_LEVEL_SYL_CURVES)
      FA_CUDA(h->g_features.reserve((Fz + nz) * h->feat_width() * sizeof(double)));
  }
  if (h->ctl_chunk > 0 && h->cfg.output_level >= 3) {
    const int CH = h->ctl_chunk;
    h->cchunk_base.assign((size_t)n + 1, 0);
    for (int i = 0; i < n; i++) h->cchunk_base[i + 1] = h->cchunk_base[i] + std::max(1, (h->utts[i].frames + CH - 1) / CH);
    h->total_cchunks = h->cchunk_base[n];
    const size_t tc = (size_t)h->total_cchunks;
    std::vector<int> lists(2 * tc);
    for (int i = 0; i < n; i++)
      for (long long c = h->cchunk_base[i]; c < h->cchunk_base[i + 1]; c++) { lists[c] = i; lists[tc + c] = (int)(c - h->cchunk_base[i]); }
    FA_CUDA(h->d_cchunks.reserve(2 * tc * sizeof(int) + ((size_t)n + 1) * sizeof(long long) + 16));
    FA_CUDA(cudaMemcpyAsync(h->d_cchunks.p, h->cchunk_base.data(), ((size_t)n + 1) * sizeof(long long), cudaMemcpyHostToDevice, s));
    FA_CUDA(cudaMemcpyAsync((char*)h->d_cchunks.p + ((size_t)n + 1) * sizeof(long long), lists.data(), 2 * tc * sizeof(int),
                            cudaMemcpyHostToDevice, s));
    FA_CUDA(cudaStreamSynchronize(s));
    FA_CUDA(h->d_cstate.reserve(2 * tc * sizeof(FaCtlState)));
    FA_CUDA(h->d_frT.reserve(Fz * sizeof(double)));
    FA_CUDA(h->d_frk.reserve(Fz * sizeof(int)));
    FA_CUDA(h->d_frthr.reserve(Fz * sizeof(double)));
  }
  FA_CUDA(h->d_fix.reserve(16));
  if (h->chunk_frames > 0) {
    const int CH = h->chunk_frames;
    h->chunk_base.assign((size_t)n + 1, 0);
    for (int i = 0; i < n; i++) h->chunk_base[i + 1] = h->chunk_base[i] + std::max(1, (h->utts[i].frames + CH - 1) / CH);
    h->total_chunks = h->chunk_base[n];
    const size_t tc = (size_t)h->total_chunks;
    std::vector<int> lists(2 * tc);
    for (int i = 0; i < n; i++)
      for (long long c = h->chunk_base[i]; c < h->chunk_base[i + 1]; c++) { lists[c] = i; lists[tc + c] = (int)(c - h->chunk_base[i]); }
    const size_t bytes = 2 * tc * sizeof(int) + ((size_t)n + 1) * sizeof(long long) + 16;
    FA_CUDA(h->d_chunks.reserve(bytes));
    // layout: base[n+1] (long long) | utt[tc] | idx[tc]
    FA_CUDA(cudaMemcpyAsync(h->d_chunks.p, h->chunk_base.data(), ((size_t)n + 1) * sizeof(long long), cudaMemcpyHostToDevice, s));
    FA_CUDA(cudaMemcpyAsync((char*)h->d_chunks.p + ((size_t)n + 1) * sizeof(long long), lists.data(), 2 * tc * sizeof(int),
                            cudaMemcpyHostToDevice, s));
    FA_CUDA(cudaStreamSynchronize(s));   // `lists` dies at scope exit
    FA_CUDA(h->d_state.reserve(2 * tc * (size_t)h->M * sizeof(float)));
    if (h->want_spec && h->spec_fmt() == FA_SPECTRUM_F32) FA_CUDA(h->d_specdb.reserve(Fz * h->M * sizeof(float)));
  }
  h->prepared = true;
  return FA_OK;
}

static int ensure_sub_streams(fa_handle* h, int n) {
  for (int i = h->n_sub_streams; i < n && i < kMaxSub; i++) {
    FA_CUDA(cudaStreamCreateWithFlags(&h->sub_stream[i], cudaStreamNonBlocking));
    if (h->k3_priority) FA_CUDA(cudaStreamCreateWithPriority(&h->sub_hi[i], cudaStreamNonBlocking, h->prio_hi));
    FA_CUDA(cudaEventCreateWithFlags(&h->sub_done[i], cudaEventDisableTiming));
    FA_CUDA(cudaEventCreateWithFlags(&h->sub_mid[i], cudaEventDisableTiming));
    FA_CUDA(cudaEventCreateWithFlags(&h->sub_hi_done[i], cudaEventDisableTiming));
    FA_CUDA(cudaEventCreateWithFlags(&h->spec_done[i], cudaEventDisableTiming));
    FA_CUDA(cudaEventCreateWithFlags(&h->copy_done[i], cudaEventDisableTiming));
    if (h->trace) for (int k = 0; k < 4; k++) FA_CUDA(cudaEventCreate(&h->tr_ev[i][k]));
    if (h->trace) for (int k = 0; k < 5; k++) FA_CUDA(cudaEventCreate(&h->tr_k[i][k]));
    h->n_sub_streams = i + 1;
  }
  return FA_OK;
}

// split the batch into sub-batches of whole utterances with about equal frame counts
static std::vector<SubBatch> plan(const fa_handle* h, bool with_copies) {
  const int n = (int)h->utts.size();
  int S = h->pipeline;
  // automatic: many sub-batches when PCIe copies have to overlap the kernels, few when the data is resident (every
  // stage but K1a is a per-utterance latency chain, so extra sub-batches only add launches)
  if (S == 0) S = with_copies ? std::min(8, std::max(1, n / 60)) : std::min(2, std::max(1, n / 250));
  S = std::max(1, std::min(S, n));
  std::vector<SubBatch> out;
  const long long F = h->total_frames;
  int u = 0;
  for (int b = 0; b < S; b++) {
    SubBatch sb;
    sb.u0 = u;
    const long long target = F * (b + 1) / S;
    if (b == S - 1) u = n;
    else {
      while (u < n && h->utts[u].row0 + h->utts[u].frames <= target) u++;
      if (u == sb.u0 && u < n) u++;
    }
    sb.u1 = u;
    sb.r0 = sb.u0 < n ? h->utts[sb.u0].row0 : F;
    sb.r1 = sb.u1 < n ? h->utts[sb.u1].row0 : F;
    if (sb.u1 > sb.u0) out.push_back(sb);
    if (u >= n) break;
  }
  return out;
}

// H2D of the PCM of utterances [u0, u1): contiguous runs per region
static int copy_pcm_range(fa_handle* h, int u0, int u1, cudaStream_t s) {
  if (h->frames_mode) {   // the input of the batch is the uint32 frames themselves
    if (u1 <= u0) return FA_OK;
    const long long r0 = h->utts[u0].row0, r1 = h->utts[u1 - 1].row0 + h->utts[u1 - 1].frames;
    const size_t row = (size_t)h->B * sizeof(uint32_t);
    if (r1 > r0)
      FA_CUDA(cudaMemcpyAsync((char*)h->d_frames.p + (size_t)r0 * row, (const char*)h->h_frames.p + (size_t)r0 * row,
                              (size_t)(r1 - r0) * row, cudaMemcpyHostToDevice, s));
    return FA_OK;
  }
  int i = u0;
  while (i < u1) {
    const int reg = h->utts[i].region;
    long long lo = h->utts[i].off, hi = lo + ((h->utts[i].n + 3) & ~3ll);
    int j = i + 1;
    while (j < u1 && h->utts[j].region == reg && h->utts[j].off >= lo) {
      hi = std::max(hi, h->utts[j].off + ((h->utts[j].n + 3) & ~3ll));
      j++;
    }
    const Region& r = h->regions[reg];
    const float* host = reg == 0 ? h->h_pcm.as<float>() : r.host;
    hi = std::min(hi, reg == 0 ? h->staged : r.n);
    if (hi > lo && r.host16) {
      int16_t* d16 = h->d_pcm16.as<int16_t>() + r.dev_off + lo;
      FA_CUDA(cudaMemcpyAsync(d16, r.host16 + lo, (size_t)(hi - lo) * sizeof(int16_t), cudaMemcpyHostToDevice, s));
      FA_CUDA(fa_launch_pcm_i16(d16, h->d_pcm.as<float>() + r.dev_off + lo, hi - lo, s, &h->launches));
    } else if (hi > lo)
      FA_CUDA(cudaMemcpyAsync(h->d_pcm.as<float>() + r.dev_off + lo, host + lo, (size_t)(hi - lo) * sizeof(float),
                              cudaMemcpyHostToDevice, s));
    i = j;
  }
  return FA_OK;
}

// stages 1-4 of one sub-batch on stream s
// (s3 != s: the segment scan + features go to the high-priority stream s3 so that their few, long-lived warps are placed
// ahead of the queued spectrum CTAs of other sub-batches / batches and run beside them)
static int launch_sub(fa_handle* h, const SubBatch& sb, int slot, cudaStream_t s, cudaEvent_t* ev /* 5 or null */,
                      cudaStream_t s3 = nullptr) {
  if (!s3) s3 = s;
  const fa_config& c = h->cfg;
  const int n = (int)h->utts.size();
  const long long F = h->total_frames;
  const long long* meta = h->d_meta.as<long long>();
  if (ev) FA_CUDA(cudaEventRecord(ev[0], s));
  const bool tr = !ev && h->trace;
  if (tr) FA_CUDA(cudaEventRecord(h->tr_k[slot][0], s));
  FaSpectrumParams sp;
  memset(&sp, 0, sizeof(sp));
  sp.pcm = h->d_pcm.as<float>();
  sp.utt_off = meta; sp.utt_len = meta + n; sp.frame_off = meta + 2 * n;
  sp.n_utt = n; sp.utt_begin = sb.u0; sp.utt_count = sb.u1 - sb.u0; sp.row_begin = sb.r0;
  sp.hop = h->hop; sp.N = h->N; sp.M = h->M; sp.logM = h->logM; sp.B = h->B;
  sp.win = h->d_win.as<float>(); sp.tw = h->d_tw.as<float2>(); sp.tw_stage = h->d_tws.as<float2>(); sp.ws = h->d_ws.as<float2>();
  sp.bm_k0 = h->d_bmi.as<int>(); sp.bm_cnt = sp.bm_k0 + h->B; sp.bm_off = sp.bm_k0 + 2 * h->B;
  sp.bm_w = h->d_bmw.as<float>(); sp.n_weights = h->n_weights;
  sp.emph = h->d_emph.as<float>(); sp.use_emph = c.high_f_emph != 0.0; sp.power = c.spec_type == FA_SPEC_POWER;
  sp.gain = fa_tab_gain(&c); sp.tau = (float)c.smoothing; sp.omt = (float)(1.0 - c.smoothing);
  sp.inv2N = (float)(1.0 / (2.0 * (double)h->N)); sp.min_db = (float)c.min_db; sp.max_db = (float)c.max_db;
  sp.clamp_db = c.clamp_db;
  sp.scratch_mag = 1;
  sp.write_db = h->want_spec;
  sp.fused = h->use_fused();
  sp.k1a_variant = h->k1a_variant;
  sp.spec_fmt = h->spec_fmt();
  sp.spec_q = h->d_specq.p;
  sp.byte_scale = (float)(255.0 / (c.max_db - c.min_db));
  sp.n_rows = sb.r1 - sb.r0;
  sp.spec_db = h->d_spec.as<float>();
  sp.frames = h->d_frames.as<uint32_t>();
  sp.work_counter = h->d_counter.as<int>() + slot;
  if (h->chunk_frames > 0) {
    const size_t tc = (size_t)h->total_chunks;
    const long long* base = h->d_chunks.as<long long>();
    const int* utt_list = reinterpret_cast<const int*>(base + n + 1);
    const long long c0 = h->chunk_base[sb.u0], c1 = h->chunk_base[sb.u1];
    sp.chunk_frames = h->chunk_frames; sp.warm_frames = h->warm_frames;
    sp.chunk_base = base; sp.chunk_utt = utt_list + c0; sp.chunk_idx = utt_list + tc + c0; sp.n_chunks = (int)(c1 - c0);
    sp.st_entry = h->d_state.as<float>(); sp.st_exit = sp.st_entry + tc * h->M;
    sp.spec_out = (h->want_spec && h->spec_fmt() == FA_SPECTRUM_F32) ? h->d_specdb.as<float>() : nullptr;
    sp.fixups = h->d_fix.as<int>();
  }
  if (!h->frames_mode) FA_CUDA(fa_launch_spectrum(sp, s, &h->launches, ev ? h->ev[7] : nullptr));
  else if (ev) FA_CUDA(cudaEventRecord(h->ev[7], s));
  if (h->debug_sync) FA_CUDA(cudaStreamSynchronize(s));
  if (ev) FA_CUDA(cudaEventRecord(ev[1], s));
  if (!ev) FA_CUDA(cudaEventRecord(h->spec_done[slot], s));  // the dB rows of this sub-batch are final
  if (!ev && h->trace) FA_CUDA(cudaEventRecord(h->tr_ev[slot][1], s));
  if (tr) FA_CUDA(cudaEventRecord(h->tr_k[slot][1], s));
  if (c.output_level >= 3 && sb.r1 > sb.r0) {
    FaPeaksParams pp;
    pp.frames = h->d_frames.as<uint32_t>(); pp.B = h->B; pp.maxp = h->maxp; pp.n_frames = sb.r1 - sb.r0; pp.row_begin = sb.r0;
    pp.cand = h->d_cand.as<FaCand>(); pp.ncand = h->d_ncand.as<int>(); pp.gsum = h->d_gsum.as<double>();
    FA_CUDA(fa_launch_peaks(pp, s, &h->launches));
    if (h->debug_sync) FA_CUDA(cudaStreamSynchronize(s));
  }
  if (ev) FA_CUDA(cudaEventRecord(ev[2], s));
  if (tr) FA_CUDA(cudaEventRecord(h->tr_k[slot][2], s));
  if (s3 != s && c.output_level >= 3) {
    FA_CUDA(cudaEventRecord(h->sub_mid[slot], s));
    FA_CUDA(cudaStreamWaitEvent(s3, h->sub_mid[slot], 0));
  }
  if (c.output_level >= 3) {
    const size_t T = (size_t)std::max<long long>(h->track_total, 1);
    const size_t P = (size_t)std::max<long long>(F, 1) * h->maxp;
    const size_t R = (size_t)std::max<long long>(F, 1) + n;
    FaSegmentParams g;
    memset(&g, 0, sizeof(g));
    g.cand = h->d_cand.as<FaCand>(); g.ncand = h->d_ncand.as<int>();
    g.gsum = h->d_gsum.as<double>(); g.frame_off = meta + 2 * n; g.n_utt = n; g.B = h->B; g.maxp = h->maxp;
    g.utt_begin = sb.u0; g.utt_count = sb.u1 - sb.u0;
    g.level = c.output_level;
    g.max_voiced_bin = (int)fa_js_parse_int(0.7 * (double)h->B);
    g.seg_min_frames = (int)fa_js_parse_int(c.min_seg_length_ms / c.window_step_ms);
    g.auto_gate = c.auto_noise_gate;
    g.seg_breaker = c.pause_length_ms > 2 * c.window_step_ms ? c.pause_length_ms / c.window_step_ms : 250 / c.window_step_ms;
    if (c.auto_noise_gate) { g.y0 = 50; g.v0 = 2; }
    else { g.y0 = fa_js_pow(10, c.voiced_max_db / 20); g.v0 = fa_js_pow(10, c.voiced_min_db / 20); }
    g.track_base = const_cast<long long*>(meta + 3 * n + 1);
    g.trk_count = h->d_trk_i.as<int>(); g.trk_order = g.trk_count + T; g.trk_rank = g.trk_order + T;
    g.trk_sum_e = h->d_trk_d.as<double>(); g.trk_sum_eb = g.trk_sum_e + T; g.trk_mean = g.trk_sum_eb + T;
    g.trk_slot = h->d_trk_slot.as<signed char>();
    g.pt_track = h->d_pt_i.as<int>(); g.pt_ord = g.pt_track + P; g.pt_frame = g.pt_ord + P; g.pt_binspan = g.pt_frame + P;
    g.pt_e = h->d_pt_e.as<double>();
    g.pt_amp = c.output_level == FA_LEVEL_SEGMENTS ? h->d_pt_amp.as<int>() : nullptr;
    g.track_points = c.output_level == FA_LEVEL_SEGMENTS ? h->d_formants.as<fa_track_point>() : nullptr;
    g.row_count = h->d_rows.as<int>(); g.row_off = g.row_count + R; g.row_list = h->d_rowlist.as<int>();
    g.cs_spill = h->d_spill.as<unsigned long long>();
    g.finalize_in_smem = h->k3_finalize_smem;
    g.no_truncate = h->no_truncate;
    g.impl = h->k3_impl; g.warps_per_cta = h->k3_warps; g.reg_cap = h->k3_regs; g.redo_count = h->d_fix.as<int>() + 2;
    g.mode = h->k3_mode;
    if (h->k3_epochs()) {
      g.epochs = h->d_epochs.as<FaEpoch>();
      g.work = h->d_work.as<int2>() + (sb.r0 + sb.u0);      // the sub-batch's slice (capacity: its frames + utterances)
      g.work_count = h->d_k3q.as<int>() + 2 * slot;
    }
    if (g.mode == 1) {
      g.fr_ctl = h->d_frctl.as<unsigned>(); g.fr_v = h->d_frv.as<double>();
      g.n_workers = h->k3_workers;
      if (h->ctl_chunk > 0) {
        const size_t tc = (size_t)h->total_cchunks;
        const long long* base = h->d_cchunks.as<long long>();
        const int* lst = reinterpret_cast<const int*>(base + n + 1);
        const long long c0 = h->cchunk_base[sb.u0], c1 = h->cchunk_base[sb.u1];
        g.ctl_chunk = h->ctl_chunk; g.ctl_warm = h->ctl_warm;
        g.cchunk_base = base; g.cchunk_utt = lst + c0; g.cchunk_idx = lst + tc + c0; g.n_cchunks = (int)(c1 - c0);
        g.ctl_entry = h->d_cstate.as<FaCtlState>(); g.ctl_exit = g.ctl_entry + tc;
        g.fr_T = h->d_frT.as<double>(); g.fr_k = h->d_frk.as<int>(); g.fr_thr = h->d_frthr.as<double>();
        g.ctl_fixups = h->d_fix.as<int>() + 1;
      }
    }
    g.segs = h->d_segs.as<fa_segment>(); g.syls = h->d_syls.as<fa_syllable>();
    g.formants = h->d_formants.as<float>(); g.energy = h->d_energy.as<float>();
    int* cnt = h->d_counts.as<int>();
    g.n_segs = cnt; g.n_stored = cnt + n; g.n_rows = cnt + 2 * n; g.n_syls = cnt + 3 * n; g.overflow = cnt + 5 * n;
    FA_CUDA(fa_launch_segment(g, s3, &h->launches));
    if (ev) FA_CUDA(cudaEventRecord(ev[3], s));
    if (tr) FA_CUDA(cudaEventRecord(h->tr_k[slot][3], s3));
    if (c.output_level == 5 || c.output_level == 13) {
      FaFeatureParams fp;
      fp.frame_off = meta + 2 * n; fp.n_utt = n; fp.level = c.output_level;
      fp.utt_begin = sb.u0; fp.utt_count = sb.u1 - sb.u0;
      fp.segs = g.segs; fp.n_segs = g.n_segs; fp.syls = g.syls; fp.n_syls = g.n_syls; fp.formants = g.formants;
      fp.features = h->d_features.as<double>(); fp.n_feat = cnt + 4 * n;
      fp.epochs = h->k3_epochs() ? h->d_epochs.as<FaEpoch>() : nullptr;
      // rows of one utterance are spread over `row_slices` CTAs (a one-hour stream has ~2000 rows in ONE utterance)
      fp.row_slices = (int)std::min<long long>(64, std::max<long long>(1, (sb.r1 - sb.r0) / std::max(1, sb.u1 - sb.u0) / 256));
      FA_CUDA(fa_launch_features(fp, s3, &h->launches));
    }
    if (c.output_level == FA_LEVEL_SYL_CURVES) {
      FaCurveParams cp;
      cp.frame_off = meta + 2 * n; cp.n_utt = n; cp.utt_begin = sb.u0; cp.utt_count = sb.u1 - sb.u0;
      cp.segs = g.segs; cp.n_segs = g.n_segs; cp.syls = g.syls; cp.n_syls = g.n_syls; cp.formants = g.formants; cp.energy = g.energy;
      cp.epochs = h->k3_epochs() ? h->d_epochs.as<FaEpoch>() : nullptr;
      cp.list = h->d_curve_list.as<int2>() + (sb.r0 + sb.u0); cp.list_count = h->d_curve_count.as<int>() + slot;
      cp.list_cap = (sb.r1 - sb.r0) / 2 + (sb.u1 - sb.u0);
      cp.work = h->d_curve_work.as<double>(); cp.status = h->d_curve_status.as<int>();
      cp.rows = h->d_features.as<double>(); cp.n_feat = cnt + 4 * n;
      FA_CUDA(fa_launch_curves(cp, s3, &h->launches));
    }
    if (c.output_level == FA_LEVEL_UTTERANCE) {
      FaUtteranceParams up;
      up.frame_off = meta + 2 * n; up.n_utt = n; up.utt_begin = sb.u0; up.utt_count = sb.u1 - sb.u0;
      up.segs = g.segs; up.n_segs = g.n_segs; up.syls = g.syls; up.formants = g.formants;
      up.epochs = h->k3_epochs() ? h->d_epochs.as<FaEpoch>() : nullptr;
      up.row_base = meta + 4 * n + 2; up.rows = h->d_features.as<double>(); up.n_feat = cnt + 4 * n; up.overflow = g.overflow;
      FA_CUDA(fa_launch_utterance(up, s3, &h->launches));
    }
    if (tr) FA_CUDA(cudaEventRecord(h->tr_k[slot][4], s3));
    if (s3 != s) FA_CUDA(cudaEventRecord(h->sub_hi_done[slot], s3));
    if (ev) FA_CUDA(cudaEventRecord(ev[4], s));
  } else if (ev) {
    FA_CUDA(cudaEventRecord(ev[3], s));
    FA_CUDA(cudaEventRecord(ev[4], s));
  }
  return FA_OK;
}

// the whole device side of a run: fork into sub-batch streams, (optional) H2D + kernels + (optional) spectrum
// sink D2H per sub-batch, join, then the dense gather
static int run_device(fa_handle* h, bool with_h2d, bool with_sink) {
  cudaStream_t s = h->stream;
  const fa_config& c = h->cfg;
  const int n = (int)h->utts.size();
  const long long* meta = h->d_meta.as<long long>();
  h->launches = 0;
  if (c.output_level >= 3) FA_CUDA(cudaMemsetAsync(h->d_counts.p, 0, sizeof(int) * 6 * (size_t)n, s));
  if (c.output_level >= 3 && h->k3_epochs()) FA_CUDA(cudaMemsetAsync(h->d_k3q.p, 0, 2 * kMaxSub * sizeof(int), s));
  if (c.output_level == FA_LEVEL_SYL_CURVES) FA_CUDA(cudaMemsetAsync(h->d_curve_count.p, 0, kMaxSub * sizeof(int), s));
  FA_CUDA(cudaMemsetAsync(h->d_fix.p, 0, 3 * sizeof(int), s));
  h->fixups[0] = h->fixups[1] = h->fixups[2] = -1;
  FA_CUDA(cudaEventRecord(h->ev[0], s));
  const std::vector<SubBatch> subs = plan(h, with_h2d || (with_sink && h->spec_sink));
  const bool sink = with_sink && h->spec_sink && h->want_spec && !h->frames_mode;
  if (sink && (size_t)h->total_frames > h->spec_sink_rows) return fail(h, FA_ERR_CAPACITY, "spectrum sink too small");
  if (subs.size() <= 1) {
    SubBatch all{0, n, 0, h->total_frames};
    if (with_h2d) { const int rc = copy_pcm_range(h, 0, n, s); if (rc != FA_OK) return rc; }
    const int rc = launch_sub(h, all, 0, s, h->ev);
    if (rc != FA_OK) return rc;
    if (sink && h->total_frames)
      FA_CUDA(cudaMemcpyAsync(h->spec_sink, h->spec_out(), (size_t)h->total_frames * h->M * h->spec_elem(), cudaMemcpyDeviceToHost, s));
  } else {
    { const int rc = ensure_sub_streams(h, (int)subs.size()); if (rc != FA_OK) return rc; }
    if (sink && !h->copy_stream) {
      if (!h->own_copy_stream) FA_CUDA(cudaStreamCreateWithFlags(&h->own_copy_stream, cudaStreamNonBlocking));
      h->copy_stream = h->own_copy_stream;
    }
    FA_CUDA(cudaEventRecord(h->fork_ev, s));
    for (size_t b = 0; b < subs.size(); b++) {
      cudaStream_t ss = h->sub_stream[b];
      FA_CUDA(cudaStreamWaitEvent(ss, h->fork_ev, 0));
      if (h->trace) FA_CUDA(cudaEventRecord(h->tr_ev[b][0], ss));
      if (with_h2d) { const int rc = copy_pcm_range(h, subs[b].u0, subs[b].u1, ss); if (rc != FA_OK) return rc; }
      const bool hi = h->k3_priority && c.output_level >= 3;
      const int rc = launch_sub(h, subs[b], (int)b, ss, nullptr, hi ? h->sub_hi[b] : nullptr);
      if (rc != FA_OK) return rc;
      if (sink && subs[b].r1 > subs[b].r0) {
        // the dB rows leave as soon as the spectrum kernels of the sub-batch are done (not behind its segment scan), on
        // the copy stream: FIFO over sub-batches -- and over batches when several handles share one copy stream
        FA_CUDA(cudaStreamWaitEvent(h->copy_stream, h->spec_done[b], 0));
        if (h->trace) FA_CUDA(cudaEventRecord(h->tr_ev[b][2], h->copy_stream));
        const size_t row_bytes = (size_t)h->M * h->spec_elem();
        FA_CUDA(cudaMemcpyAsync((char*)h->spec_sink + (size_t)subs[b].r0 * row_bytes, h->spec_out() + (size_t)subs[b].r0 * row_bytes,
                                (size_t)(subs[b].r1 - subs[b].r0) * row_bytes, cudaMemcpyDeviceToHost, h->copy_stream));
        FA_CUDA(cudaEventRecord(h->copy_done[b], h->copy_stream));
        if (h->trace) FA_CUDA(cudaEventRecord(h->tr_ev[b][3], h->copy_stream));
      }
      if (hi) FA_CUDA(cudaStreamWaitEvent(ss, h->sub_hi_done[b], 0));
      FA_CUDA(cudaEventRecord(h->sub_done[b], ss));
    }
    for (size_t b = 0; b < subs.size(); b++) {
      FA_CUDA(cudaStreamWaitEvent(s, h->sub_done[b], 0));
      if (sink && subs[b].r1 > subs[b].r0) FA_CUDA(cudaStreamWaitEvent(s, h->copy_done[b], 0));
    }
    for (int i = 1; i <= 4; i++) FA_CUDA(cudaEventRecord(h->ev[i], s));  // per-stage times only exist in serial mode
    FA_CUDA(cudaEventRecord(h->ev[7], s));
  }
  if (c.output_level >= 3) {
    int* cnt = h->d_counts.as<int>();
    FaGatherArgs ga;
    ga.feat_width = h->feat_width();
    ga.l3_mult = c.output_level == FA_LEVEL_SEGMENTS ? h->maxp : 0;
    ga.epochs = h->k3_epochs() ? h->d_epochs.as<FaEpoch>() : nullptr;
    ga.row_slices = (int)std::min<long long>(64, std::max<long long>(1, h->total_frames / std::max(1, n) / 256));
    ga.feat_base = c.output_level == FA_LEVEL_UTTERANCE ? meta + 4 * n + 2 : nullptr;
    ga.frame_off = meta + 2 * n; ga.n_utt = n; ga.n_segs = cnt; ga.n_rows = cnt + 2 * n; ga.n_syls = cnt + 3 * n;
    ga.n_feat = cnt + 4 * n; ga.off = h->d_off.as<long long>();
    ga.segs = h->d_segs.as<fa_segment>(); ga.syls = h->d_syls.as<fa_syllable>();
    ga.formants = h->d_formants.as<float>(); ga.energy = h->d_energy.as<float>();
    ga.features = h->d_features.as<double>();
    ga.d_segs = h->g_segs.as<fa_segment>(); ga.d_syls = h->g_syls.as<fa_syllable>();
    ga.d_formants = h->g_formants.as<float>(); ga.d_energy = h->g_energy.as<float>();
    ga.d_features = h->g_features.as<double>();
    FA_CUDA(fa_launch_prefix(ga, s, &h->launches));
    FA_CUDA(fa_launch_gather(ga, s, &h->launches));
  }
  FA_CUDA(cudaEventRecord(h->ev[5], s));
  h->ran = true;
  h->downloaded = false;
  return FA_OK;
}

int fa_upload(fa_handle* h) {
  if (!h) return FA_ERR_INVALID_ARG;
  cudaSetDevice(h->device);
  int rc = prepare(h);
  if (rc != FA_OK) return rc;
  rc = copy_pcm_range(h, 0, (int)h->utts.size(), h->stream);
  if (rc != FA_OK) return rc;
  h->uploaded = true;
  h->ran = false;
  h->downloaded = false;
  return FA_OK;
}

int fa_run_resident(fa_handle* h) {
  if (!h) return FA_ERR_INVALID_ARG;
  if (!h->uploaded) return fail(h, FA_ERR_NOT_RUN, "fa_run_resident before fa_upload");
  cudaSetDevice(h->device);
  h->from_host = false;
  return run_device(h, false, false);
}

int fa_download(fa_handle* h) {
  if (!h) return FA_ERR_INVALID_ARG;
  if (!h->ran) return fail(h, FA_ERR_NOT_RUN, "fa_download before a run");
  cudaSetDevice(h->device);
  cudaStream_t s = h->stream;
  const int n = (int)h->utts.size();
  for (int k = 0; k < 4; k++) h->tot[k] = 0;
  if (h->cfg.output_level >= 3) {
    FA_CUDA(h->h_counts.reserve(sizeof(int) * 6 * (size_t)n));
    FA_CUDA(h->h_off.reserve(sizeof(long long) * 4 * ((size_t)n + 1)));
    FA_CUDA(cudaMemcpyAsync(h->h_counts.p, h->d_counts.p, sizeof(int) * 6 * (size_t)n, cudaMemcpyDeviceToHost, s));
    FA_CUDA(cudaMemcpyAsync(h->h_off.p, h->d_off.p, sizeof(long long) * 4 * ((size_t)n + 1), cudaMemcpyDeviceToHost, s));
    FA_CUDA(cudaStreamSynchronize(s));
    const long long* off = h->h_off.as<long long>();
    for (int k = 0; k < 4; k++) h->tot[k] = off[(size_t)k * (n + 1) + n];
    // the dense tables themselves come on demand (fetch_table): a Syllable-Features caller never pays for the formant rows
  }
  for (bool& b : h->have_table) b = false;
  FA_CUDA(cudaEventRecord(h->ev[6], s));
  h->downloaded = true;
  return FA_OK;
}

int fa_run(fa_handle* h) {
  if (!h) return FA_ERR_INVALID_ARG;
  if (h->ran) return fail(h, FA_ERR_BUSY, "Error: Already playing");
  cudaSetDevice(h->device);
  int rc = prepare(h);
  if (rc != FA_OK) return rc;
  h->uploaded = true;
  h->from_host = true;
  // asynchronous: nothing here waits for the device, so several handles can be driven from one host thread (batch i+1's
  // H2D and kernels overlap batch i's spectrum D2H); the dense result tables are fetched by fa_sync
  return run_device(h, true, true);
}

int fa_sync(fa_handle* h) {
  if (!h) return FA_ERR_INVALID_ARG;
  cudaSetDevice(h->device);
  FA_CUDA(cudaStreamSynchronize(h->stream));
  if (h->ran) {
    for (int i = 0; i < 4; i++) cudaEventElapsedTime(&h->stage_ms[i], h->ev[i], h->ev[i + 1]);
    cudaEventElapsedTime(&h->stage_ms[4], h->ev[0], h->ev[5]);
    if (cudaEventElapsedTime(&h->fft_ms, h->ev[0], h->ev[7]) != cudaSuccess || h->fft_ms > h->stage_ms[0]) {
      cudaGetLastError();
      h->fft_ms = 0.f;   // no split available (sub-batch pipeline): everything counts as the second part
    }
    if (h->trace && !h->from_host) {
      static cudaEvent_t base = nullptr;   // first traced run of the process: the common time origin of all handles
      if (!base) base = h->ev[0];
      for (int b = 0; b < h->n_sub_streams; b++) {
        float t[5];
        bool ok = true;
        for (int k = 0; k < 5; k++) ok = ok && cudaEventElapsedTime(&t[k], base, h->tr_k[b][k]) == cudaSuccess;
        cudaGetLastError();
        if (ok) fprintf(stderr, "FA_TRACE_K h=%p sub=%d start=%.3f spectrum_end=%.3f peaks_end=%.3f segment_end=%.3f features_end=%.3f\n",
                        (void*)h, b, t[0], t[1], t[2], t[3], t[4]);
      }
    }
    if (h->trace && h->from_host) {
      for (int b = 0; b < h->n_sub_streams; b++) {
        float t[4] = {-1, -1, -1, -1};
        bool ok = true;
        for (int k = 0; k < 4; k++) ok = ok && cudaEventElapsedTime(&t[k], h->ev[0], h->tr_ev[b][k]) == cudaSuccess;
        cudaGetLastError();
        if (ok) fprintf(stderr, "FA_TRACE h=%p run=%d sub=%d start=%.3f spec_done=%.3f d2h_start=%.3f d2h_end=%.3f total=%.3f\n",
                        (void*)h, h->trace_seq, b, t[0], t[1], t[2], t[3], h->stage_ms[4]);
      }
      h->trace_seq++;
    }
    if (h->from_host && !h->downloaded) {  // fa_run: the table sizes are known now; fetch the dense tables
      const int rc = fa_download(h);
      if (rc != FA_OK) return rc;
      FA_CUDA(cudaStreamSynchronize(h->stream));
    }
  }
  return FA_OK;
}

int fa_stage_times(fa_handle* h, float ms[5]) {
  if (!h || !ms) return FA_ERR_INVALID_ARG;
  if (!h->ran) return fail(h, FA_ERR_NOT_RUN, "no run yet");
  const int rc = fa_sync(h);
  if (rc != FA_OK) return rc;
  for (int i = 0; i < 5; i++) ms[i] = h->stage_ms[i];
  return FA_OK;
}

int fa_spectrum_split_times(fa_handle* h, float ms[2]) {
  if (!h || !ms) return FA_ERR_INVALID_ARG;
  if (!h->ran) return fail(h, FA_ERR_NOT_RUN, "no run yet");
  const int rc = fa_sync(h);
  if (rc != FA_OK) return rc;
  ms[0] = h->fft_ms;
  ms[1] = h->stage_ms[0] - h->fft_ms;
  return FA_OK;
}

int fa_launch_count(fa_handle* h) { return h ? h->launches : FA_ERR_INVALID_ARG; }

int fa_stream_fixups(fa_handle* h, int stage) {
  if (!h || stage < 0 || stage > 2) return FA_ERR_INVALID_ARG;
  if (!h->ran) return fail(h, FA_ERR_NOT_RUN, "no run yet");
  if (h->fixups[0] < 0) {
    cudaSetDevice(h->device);
    int v[3] = {0, 0, 0};
    FA_CUDA(cudaMemcpyAsync(v, h->d_fix.p, 3 * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    FA_CUDA(cudaStreamSynchronize(h->stream));
    h->fixups[0] = v[0]; h->fixups[1] = v[1]; h->fixups[2] = v[2];
  }
  return h->fixups[stage];
}
int fa_num_utterances(const fa_handle* h) { return h ? (int)h->utts.size() : FA_ERR_INVALID_ARG; }

static int need_results(fa_handle* h) {
  if (!h) return FA_ERR_INVALID_ARG;
  if (!h->ran) return fail(h, FA_ERR_NOT_RUN, "results requested before fa_run");
  cudaSetDevice(h->device);
  if (!h->downloaded) {
    const int rc = fa_download(h);
    if (rc != FA_OK) return rc;
  }
  cudaError_t e = cudaStreamSynchronize(h->stream);
  if (e != cudaSuccess) return fail(h, FA_ERR_CUDA, "sync", e);
  return FA_OK;
}

// whole-batch results are only handed out when no utterance overflowed an internal table (their tables are partial)
static int batch_overflow(fa_handle* h) {
  if (h->cfg.output_level < 3) return 0;
  const int n = (int)h->utts.size();
  const int* k = h->h_counts.as<int>() + 5 * (size_t)n;
  int bad = 0;
  for (int i = 0; i < n; i++) bad += k[i] != 0;
  return bad;
}

static void fill_counts(fa_handle* h, int i, fa_counts* c) {
  const Utt& u = h->utts[i];
  const int n = (int)h->utts.size();
  memset(c, 0, sizeof(*c));
  c->samples = u.n; c->sample_rate = h->sample_rate; c->hop = h->hop; c->frames = u.frames; c->bands = h->B;
  if (h->cfg.output_level >= 3) {
    const int* k = h->h_counts.as<int>();
    c->segments = k[i]; c->stored_segments = k[n + i]; c->formant_rows = k[2 * n + i]; c->syllables = k[3 * n + i];
    c->feature_rows = k[4 * n + i]; c->overflow = k[5 * n + i];
  }
}

int fa_result_counts(fa_handle* h, int64_t utt_id, fa_counts* out) {
  int rc = need_results(h);
  if (rc != FA_OK) return rc;
  if (!out) return FA_ERR_INVALID_ARG;
  Utt* u = find_utt(h, utt_id);
  if (!u) return fail(h, FA_ERR_UNKNOWN_UTT, "unknown utterance id");
  fill_counts(h, (int)(u - h->utts.data()), out);
  return out->overflow ? fail(h, FA_ERR_CAPACITY, "an internal table overflowed for this utterance") : FA_OK;
}

int fa_total_counts(fa_handle* h, fa_counts* out) {
  int rc = need_results(h);
  if (rc != FA_OK) return rc;
  if (!out) return FA_ERR_INVALID_ARG;
  memset(out, 0, sizeof(*out));
  out->sample_rate = h->sample_rate; out->hop = h->hop; out->bands = h->B;
  for (size_t i = 0; i < h->utts.size(); i++) {
    fa_counts c;
    fill_counts(h, (int)i, &c);
    out->samples += c.samples; out->frames += c.frames; out->segments += c.segments;
    out->stored_segments += c.stored_segments; out->formant_rows += c.formant_rows; out->syllables += c.syllables;
    out->feature_rows += c.feature_rows; out->overflow += c.overflow;
  }
  return out->overflow ? fail(h, FA_ERR_CAPACITY, "an internal table overflowed for at least one utterance of the batch") : FA_OK;
}

int fa_copy_counts_table(fa_handle* h, fa_counts* dst, size_t cap) {
  int rc = need_results(h);
  if (rc != FA_OK) return rc;
  const size_t n = h->utts.size();
  if (n > cap) return fail(h, FA_ERR_CAPACITY, "destination too small");
  if (n && !dst) return FA_ERR_INVALID_ARG;
  for (size_t i = 0; i < n; i++) fill_counts(h, (int)i, dst + i);
  return (int)n;
}

// rows of utterance `utt_id` (or of the whole batch when utt_id < 0) from a device table with a fixed row size
static int copy_rows_device(fa_handle* h, int64_t utt_id, const void* dev, size_t row_bytes, void* dst, size_t cap_rows) {
  int rc = need_results(h);
  if (rc != FA_OK) return rc;
  long long r0 = 0, nr = h->total_frames;
  if (utt_id >= 0) {
    Utt* u = find_utt(h, utt_id);
    if (!u) return fail(h, FA_ERR_UNKNOWN_UTT, "unknown utterance id");
    r0 = u->row0; nr = u->frames;
  }
  if ((size_t)nr > cap_rows) return fail(h, FA_ERR_CAPACITY, "destination too small");
  if (nr == 0) return 0;
  if (!dst) return FA_ERR_INVALID_ARG;
  FA_CUDA(cudaMemcpyAsync(dst, (const char*)dev + (size_t)r0 * row_bytes, (size_t)nr * row_bytes, cudaMemcpyDeviceToHost, h->stream));
  FA_CUDA(cudaStreamSynchronize(h->stream));
  return (int)nr;
}

int fa_copy_spectrum_raw(fa_handle* h, int64_t utt_id, void* dst, size_t cap_rows) {
  if (!h) return FA_ERR_INVALID_ARG;
  if (!h->want_spec) return fail(h, FA_ERR_INVALID_ARG, "spectrum not materialised (set want_spectrum or output_level <= 2)");
  if (h->frames_mode) return fail(h, FA_ERR_INVALID_ARG, "spectrum not materialised (the batch was submitted as frames)");
  return copy_rows_device(h, utt_id, h->spec_out(), (size_t)h->M * h->spec_elem(), dst, cap_rows);
}

int fa_copy_spectrum(fa_handle* h, int64_t utt_id, float* dst, size_t cap_rows) {
  if (!h) return FA_ERR_INVALID_ARG;
  if (h->spec_fmt() != FA_SPECTRUM_F32) return fail(h, FA_ERR_INVALID_ARG, "spectrum_format is not float32: use fa_copy_spectrum_raw");
  return fa_copy_spectrum_raw(h, utt_id, dst, cap_rows);
}

int fa_copy_frames(fa_handle* h, int64_t utt_id, uint32_t* dst, size_t cap_rows) {
  if (!h) return FA_ERR_INVALID_ARG;
  return copy_rows_device(h, utt_id, h->d_frames.p, (size_t)h->B * sizeof(uint32_t), dst, cap_rows);
}

// one dense table device -> pinned host, once per run: 0 segs, 1 formants, 2 energy, 3 syls, 4 features
static int fetch_table(fa_handle* h, int table) {
  if (h->have_table[table] || h->cfg.output_level < 3) return FA_OK;
  cudaStream_t s = h->stream;
  HostBuf* hb[5] = {&h->h_segs, &h->h_formants, &h->h_energy, &h->h_syls, &h->h_features};
  DevBuf* db[5] = {&h->g_segs, &h->g_formants, &h->g_energy, &h->g_syls, &h->g_features};
  const size_t rows = (size_t)h->tot[table == 0 ? 0 : table <= 2 ? 1 : table == 3 ? 2 : 3];
  if (h->cfg.output_level == FA_LEVEL_SEGMENTS && table == 2) { h->have_table[table] = true; return FA_OK; }   // no energy rows
  const size_t row_bytes = table == 0 ? sizeof(fa_segment) : table == 1 ? h->row_bytes() : table == 2 ? 3 * sizeof(float)
                           : table == 3 ? sizeof(fa_syllable) : (size_t)h->feat_width() * sizeof(double);
  FA_CUDA(hb[table]->reserve(std::max<size_t>(16, rows * row_bytes)));
  if (rows) {
    FA_CUDA(cudaMemcpyAsync(hb[table]->p, db[table]->p, rows * row_bytes, cudaMemcpyDeviceToHost, s));
    FA_CUDA(cudaStreamSynchronize(s));
  }
  h->have_table[table] = true;
  return FA_OK;
}

// dense host tables: kind 0 segs, 1 rows, 2 syls, 3 feat (offset tables); table: see fetch_table
static int copy_dense(fa_handle* h, int64_t utt_id, int kind, int table, size_t row_bytes, void* dst, size_t cap_rows) {
  int rc = need_results(h);
  if (rc != FA_OK) return rc;
  if (h->cfg.output_level < 3) return 0;
  rc = fetch_table(h, table);
  if (rc != FA_OK) return rc;
  HostBuf* hb[5] = {&h->h_segs, &h->h_formants, &h->h_energy, &h->h_syls, &h->h_features};
  const void* host = hb[table]->p;
  const int n = (int)h->utts.size();
  const long long* off = h->h_off.as<long long>() + (size_t)kind * (n + 1);
  long long r0 = 0, nr = off[n];
  if (utt_id >= 0) {
    Utt* u = find_utt(h, utt_id);
    if (!u) return fail(h, FA_ERR_UNKNOWN_UTT, "unknown utterance id");
    const int i = (int)(u - h->utts.data());
    if (h->h_counts.as<int>()[5 * n + i]) return fail(h, FA_ERR_CAPACITY, "an internal table overflowed for this utterance");
    r0 = off[i]; nr = off[i + 1] - off[i];
  } else if (batch_overflow(h)) return fail(h, FA_ERR_CAPACITY, "an internal table overflowed for at least one utterance of the batch");
  if ((size_t)nr > cap_rows) return fail(h, FA_ERR_CAPACITY, "destination too small");
  if (nr && !dst) return FA_ERR_INVALID_ARG;
  if (nr) memcpy(dst, (const char*)host + (size_t)r0 * row_bytes, (size_t)nr * row_bytes);
  return (int)nr;
}

int fa_set_truncate(fa_handle* h, int on) {
  if (!h) return FA_ERR_INVALID_ARG;
  h->no_truncate = on ? 0 : 1;
  return FA_OK;
}

int fa_copy_segments(fa_handle* h, int64_t utt_id, fa_segment* dst, size_t cap) {
  if (!h) return FA_ERR_INVALID_ARG;
  return copy_dense(h, utt_id, 0, 0, sizeof(fa_segment), dst, cap);
}
int fa_copy_formants(fa_handle* h, int64_t utt_id, float* dst, size_t cap) {
  if (!h) return FA_ERR_INVALID_ARG;
  if (h->cfg.output_level == FA_LEVEL_SEGMENTS) return 0;   // level 3 stores no straightened rows (fa_copy_track_points)
  return copy_dense(h, utt_id, 1, 1, 9 * sizeof(float), dst, cap);
}
int fa_copy_track_points(fa_handle* h, int64_t utt_id, fa_track_point* dst, size_t cap) {
  if (!h) return FA_ERR_INVALID_ARG;
  if (h->cfg.output_level != FA_LEVEL_SEGMENTS) return fail(h, FA_ERR_INVALID_ARG, "raw tracks need output_level 3");
  return copy_dense(h, utt_id, 1, 1, sizeof(fa_track_point), dst, cap);
}
int fa_copy_energy(fa_handle* h, int64_t utt_id, float* dst, size_t cap) {
  if (!h) return FA_ERR_INVALID_ARG;
  if (h->cfg.output_level == FA_LEVEL_SEGMENTS) return 0;
  return copy_dense(h, utt_id, 1, 2, 3 * sizeof(float), dst, cap);
}
int fa_copy_syllables(fa_handle* h, int64_t utt_id, fa_syllable* dst, size_t cap) {
  if (!h) return FA_ERR_INVALID_ARG;
  return copy_dense(h, utt_id, 2, 3, sizeof(fa_syllable), dst, cap);
}
int fa_copy_features(fa_handle* h, int64_t utt_id, double* dst, size_t cap) {
  if (!h) return FA_ERR_INVALID_ARG;
  if (h->cfg.output_level == FA_LEVEL_UTTERANCE)
    return fail(h, FA_ERR_INVALID_ARG, "level 11 rows have 264 entries: use fa_copy_utterance_features");
  if (h->cfg.output_level == FA_LEVEL_SYL_CURVES)
    return fail(h, FA_ERR_INVALID_ARG, "level 12 rows have 23 entries: use fa_copy_curve_features");
  return copy_dense(h, utt_id, 3, 4, FA_N_FEATURES * sizeof(double), dst, cap);
}

int fa_copy_curve_features(fa_handle* h, int64_t utt_id, double* dst, size_t cap) {
  if (!h) return FA_ERR_INVALID_ARG;
  if (h->cfg.output_level != FA_LEVEL_SYL_CURVES) return fail(h, FA_ERR_INVALID_ARG, "syllable curves need output_level 12");
  return copy_dense(h, utt_id, 3, 4, FA_N_CURVE_FEATURES * sizeof(double), dst, cap);
}

int fa_copy_utterance_features(fa_handle* h, int64_t utt_id, double* dst, size_t cap) {
  if (!h) return FA_ERR_INVALID_ARG;
  if (h->cfg.output_level != FA_LEVEL_UTTERANCE) return fail(h, FA_ERR_INVALID_ARG, "utterance distributions need output_level 11");
  return copy_dense(h, utt_id, 3, 4, FA_N_UTT_FEATURES * sizeof(double), dst, cap);
}

int fa_mlp_classify_features(fa_mlp* m, fa_handle* h, int64_t utt_id, float* probs, size_t cap_rows) {
  if (!m || !h) return FA_ERR_INVALID_ARG;
  const int lvl = h->cfg.output_level;
  if (lvl != FA_LEVEL_SEG_FEATURES && lvl != FA_LEVEL_SYL_FEATURES && lvl != FA_LEVEL_UTTERANCE)
    return fail(h, FA_ERR_INVALID_ARG, "no feature rows at this output_level");
  if (fa_mlp_in_dim(m) != h->feat_width()) return fail(h, FA_ERR_INVALID_ARG, "model input width != feature row width");
  if (fa_mlp_device(m) != h->device) return fail(h, FA_ERR_INVALID_ARG, "the model and the handle live on different devices");
  int rc = need_results(h);
  if (rc != FA_OK) return rc;
  const int n = (int)h->utts.size();
  const long long* off = h->h_off.as<long long>() + (size_t)3 * (n + 1);
  long long r0 = 0, nr = off[n];
  if (utt_id >= 0) {
    Utt* u = find_utt(h, utt_id);
    if (!u) return fail(h, FA_ERR_UNKNOWN_UTT, "unknown utterance id");
    const int i = (int)(u - h->utts.data());
    if (h->h_counts.as<int>()[5 * n + i]) return fail(h, FA_ERR_CAPACITY, "an internal table overflowed for this utterance");
    r0 = off[i]; nr = off[i + 1] - off[i];
  } else if (batch_overflow(h)) return fail(h, FA_ERR_CAPACITY, "an internal table overflowed for at least one utterance of the batch");
  if ((size_t)nr > cap_rows) return fail(h, FA_ERR_CAPACITY, "destination too small");
  if (nr == 0) return 0;
  if (!probs) return FA_ERR_INVALID_ARG;
  // the dense feature table is still on the device (g_features): classify it in place, only the class scores come back
  rc = fa_mlp_run_device(m, h->g_features.as<double>() + (size_t)r0 * h->feat_width(), (int)nr, probs, h->stream);
  if (rc < 0) return fail(h, rc, fa_mlp_last_error(m));
  return (int)nr;
}

int fa_copy_peak_candidates(fa_handle* h, int64_t utt_id, uint32_t* packed, int32_t* counts, size_t cap_rows,
                            int32_t* max_per_frame) {
  if (!h) return FA_ERR_INVALID_ARG;
  if (h->cfg.output_level < 3) return fail(h, FA_ERR_INVALID_ARG, "no peak scan below output_level 3");
  if (max_per_frame) *max_per_frame = h->maxp;
  // the packed word of every 32-byte candidate record
  int rc = need_results(h);
  if (rc != FA_OK) return rc;
  {
    long long r0 = 0, nr = h->total_frames;
    if (utt_id >= 0) {
      Utt* u = find_utt(h, utt_id);
      if (!u) return fail(h, FA_ERR_UNKNOWN_UTT, "unknown utterance id");
      r0 = u->row0; nr = u->frames;
    }
    if ((size_t)nr > cap_rows) return fail(h, FA_ERR_CAPACITY, "destination too small");
    if (nr && !packed) return FA_ERR_INVALID_ARG;
    if (nr) {
      FA_CUDA(cudaMemcpy2DAsync(packed, sizeof(uint32_t), h->d_cand.as<FaCand>() + (size_t)r0 * h->maxp, sizeof(FaCand),
                                sizeof(uint32_t), (size_t)nr * h->maxp, cudaMemcpyDeviceToHost, h->stream));
      FA_CUDA(cudaStreamSynchronize(h->stream));
    }
  }
  return copy_rows_device(h, utt_id, h->d_ncand.p, sizeof(int), counts, cap_rows);
}

int fa_copy_gsum(fa_handle* h, int64_t utt_id, double* dst, size_t cap_rows) {
  if (!h) return FA_ERR_INVALID_ARG;
  if (h->cfg.output_level < 3) return fail(h, FA_ERR_INVALID_ARG, "no peak scan below output_level 3");
  return copy_rows_device(h, utt_id, h->d_gsum.p, sizeof(double), dst, cap_rows);
}

}  // extern "C"
