// fa_segment.cu -- K3: the per-utterance sequential scan (stages S2b, S3, S3b, S3c).
//
// Restates, for one utterance per warp (utterances are independent: reset_segmentation @B25053),
//   D()  voiced/pause decision + segment state machine   /root/reference/dist/main.js:2@B26571, @B26663
//   C()  adaptive noise gate                              @B28506
//   L()  segment reset                                    @B25649
//   O()  segment finalisation                             @B27088
//   accumulate_fm + score                                 @B35952, @B37340
//   get_ranked_formants / straighten_formants             @B35670, @B35074
//   sep_syllables                                         @B34757
// The state machine is strictly sequential in time (the threshold v of frame t depends on frame
// t-1), so the time loop is serial and the kernel is LATENCY bound: with ~2 warps per scheduler what
// matters is the dependent instruction chain per frame and -- measured with ncu -- the size of the
// hot loop (instruction-fetch stalls were 29 % of the issue slots of an unrolled variant).  Hence:
//   * K2 hands over, per candidate peak, its amplitude e[pk] and the exact prefix sums P[lo-1],
//     P[hi] of the frame, so this kernel never touches the uint32 frame: the bandwidth energy of a
//     (merged) peak is max(P[hi]) - min(P[lo-1]);
//   * candidates live one per lane; the gate filter and the (n, d, h, p) statistics are single
//     redux.sync / ballot instructions;
//   * live tracks sit in shared memory in fixed slots, lane per slot, 32 slots per pass (one pass
//     covers the usual <= 32 live tracks); expired tracks free their slot, new tracks take free slots,
//     no compaction.  Track order only matters for score ties (the reference keeps the earlier
//     track: strict '>' @B35952), which the creation index resolves;
//   * ownership of a peak = shared-memory atomicMax on the score bits, then atomicMin on the creation
//     index among the exact ties;
//   * every track update is written through to the track table / point pool in HBM (fire and forget),
//     so finalisation needs no flush;
//   * one compact code path (run-time loops over the slot passes, nothing unrolled four-fold).
// All decisions are integer compares or IEEE double arithmetic without contraction (--fmad=false)
// and the V8-equivalent log10/pow of include/fa_jsmath.h, so boundaries are bit-exact against
// oracle/fa_oracle.c.
//
// This kernel moves kilobytes per utterance; it is latency bound, not HBM bound (DESIGN.md).
#include <cstddef>
#include <cstdlib>

#include "fa_internal.cuh"
#include "fa_jsmath.h"

namespace {

constexpr int kWarps = 2;
constexpr int ACAP = 128;  // live-track slots per utterance (tracks with lastFrame >= c_ci - 3)
constexpr int PCAP = 136;  // accepted peaks per frame (>= maxp = B/2 + 4)
constexpr int CMAX = 9;    // a +-8 bin window holds at most 9 peaks (they are >= 2 bins apart)
constexpr unsigned FULL = 0xffffffffu;
constexpr int BIG = 0x7fffffff;

constexpr int CSM = 3;     // candidate scores per slot kept in shared memory; the rest spill to the point-pool tail

struct WarpShared {
  // ---- live across a finalisation ----
  uint32_t pmask[FA_MAX_BANDS / 32 + 1];      // bit b: an accepted peak has pk == b (all zero between frames)
  uint32_t pad0[3];
  uint32_t wmask[2][FA_MAX_BANDS];            // K3 v2: [set][bin] lanes whose track slot holds the peak at `bin` in its window
                                              // (all zero between frames)
  // ---- everything from here to the end of the warp's shared-memory slice is dead while a segment is finalised:
  //      finalize_fast uses it as scratch ----
  // accepted peaks of the frame
  ulonglong2 plh[PCAP];                       // P[lo-1], P[hi]
  uint2 pa[PCAP];                             // packed lo | hi<<8 | pk<<16 | last<<24, amplitude e[pk]
  unsigned long long best[PCAP];              // best score per peak (bit pattern of a positive double)
  int owner[PCAP];                            // creation index of the owning track, BIG = none
  // live tracks of the current segment (field list of l[r] @B35952)
  double t_vel[ACAP], t_se[ACAP], t_seb[ACAP];
  int t_id[ACAP];                             // creation index inside the segment, -1 = free slot
  int t_lf[ACAP];                             // lastFrame
  int t_bins[ACAP];                           // last three peak bins: b1 | b2 << 8 | b3 << 16
  int t_np[ACAP];                             // points so far
  uint32_t t_amp[ACAP];                       // lastAmp
  uint32_t t_wm[ACAP];                        // this frame: retained candidates (bit j = bin wlo + j); v2: peak lanes per owner
  unsigned char pidx[FA_MAX_BANDS];           // index of the accepted peak at bin b in the accepted list
  unsigned char newlist[PCAP];                // un-owned peaks above the gate, in peak order
  unsigned char pad1[8];
  // ---- only the general kernel (accumulate_fm) from here on: fa_segment2_kernel's slice ends in front of it (kSlimBytes) ----
  unsigned long long cs[CSM][ACAP];           // [j][slot]: score of the slot's j-th retained candidate
};
static_assert(offsetof(WarpShared, plh) % 16 == 0 && offsetof(WarpShared, cs) % 16 == 0 && sizeof(WarpShared) % 16 == 0,
              "16-byte aligned slices");
constexpr int kScratchOff = (int)offsetof(WarpShared, plh);
constexpr int kSlimBytes = (int)offsetof(WarpShared, cs);   // what accumulate_fm2 + finalize_fast touch: 3 KB less per warp


struct ScanState {
  int current_frame, no_fm_segs, c_ci, c_started, w, k;
  double y, v, x, v0, T, s_energy, c_energy;
  int n_tr, n_pts, n_slots;   // n_slots: high-water mark of used track slots (multiple passes of 32 beyond 32)
  int n_segs, n_stored, n_rows, n_syls;
  int overflow;
};

struct Bases {
  long long row0;   // first frame row of the utterance
  long long tb;     // track table base
  long long pb;     // point pool base
  long long sb;     // segment / syllable base (row0 + u)
  long long rb;     // row-scratch base (row_count / row_off)
  int F, tcap, u;
  int spill;        // slice of cs_spill (utterance in the serial kernel, worker warp in the epoch-parallel one)
};

__device__ __forceinline__ unsigned long long warp_sum_u64(unsigned long long v) {
  // exact: four 16-bit digit sums (each < 2^21) recombined
  const unsigned lo = (unsigned)v, hi = (unsigned)(v >> 32);
  const unsigned long long s0 = __reduce_add_sync(FULL, lo & 0xffffu), s1 = __reduce_add_sync(FULL, lo >> 16);
  const unsigned long long s2 = __reduce_add_sync(FULL, hi & 0xffffu), s3 = __reduce_add_sync(FULL, hi >> 16);
  return s0 + (s1 << 16) + (s2 << 32) + (s3 << 48);
}

// _() @B37340
__device__ __forceinline__ double fm_score(int gap, double dist, int count, int bin_old, int bin_new, double amp_old,
                                           double amp_new, double velocity) {
  // s = amp_new / amp_old when amp_old >= amp_new, else amp_old / amp_new (the reference's "amp_new <= 0 -> 0" exit is dead
  // there: amp_new > amp_old >= 0): ONE division of the smaller by the larger amplitude instead of two divergent ones.
  // Amplitudes are uint32 values (never NaN); 0 / 0 stays NaN and fails every test below exactly as in the reference.
  const double s_num = amp_old >= amp_new ? amp_new : amp_old, s_den = amp_old >= amp_new ? amp_old : amp_new;
  double s = s_num / s_den;
  if (gap == 0) return s > 0.1 ? 300.0 * s / dist : 0;
  if (s < 0.001) return 0;
  if (s >= 1) s = 10; else if (s < 0.1) s = 1; else s *= 10;
  double t = 10.0 - fabs((double)bin_new - (double)bin_old - velocity);
  if (t < 0) return 0;
  if (t < 1) t = 1;
  const int i = count > 10 ? 10 : count;
  // 10 / gap for gap in {1, 2, 3}: the correctly rounded quotients
  const double f = gap == 1 ? 10.0 : gap == 2 ? 5.0 : 10.0 / 3.0;
  return f * (t * t + (double)i * s);
}

// L() @B25649 (+ clear_fm @B35919)
__device__ __forceinline__ void seg_reset(ScanState& st, WarpShared& S, int started, const int lane) {
  st.c_ci = 0;
  st.c_started = started;
  st.no_fm_segs = 0;
  st.n_tr = 0;
  st.n_pts = 0;
  st.s_energy = 0.0;
  st.c_energy = 0.0;
  for (int r = lane; r < st.n_slots; r += 32) S.t_id[r] = -1;
  st.n_slots = 0;
  __syncwarp();
}

// C() @B28506 without the track reset: returns true when the gate asks for L(0).
// Only reached with the automatic gate, where e, y, x, v, v0, T are integer-valued doubles far below 2^53 (amplitudes are
// uint32, every update is a parseInt) -- so the reference's quotient tests are decided exactly by integer-exact products
// instead of FP64 divisions (a correctly rounded q = a/b with |a/b - c| >= 1/b >> ulp(c) compares with c like a/b does):
//   e > x/100  <=>  100 e > x        T/k < 30 v  <=>  T < 30 v k        v > v0/10  <=>  10 v > v0
//   parseInt(v0/20) = floor(v0/20)   (v0 < 2^32: unsigned division by a constant)
// flags: bit 0 = the T/k test asked for L(0), bit 1 = the test was evaluated; Tb, kb = T and k in front of the test
// v(y) of C() @B28506: fdlibm log10 + pow, a few thousand instructions when inlined -- and only reached when the gate's maximum
// moves.  Out of line: it keeps the scan kernels' hot loops inside the instruction cache.
__device__ __noinline__ double gate_v_of_y(const double y) {
  const double t = fa_js_log10(y);
  if (t > 7) return fa_js_parse_int(fa_js_pow(10, t - 3) / 20);
  if (t > 6) return fa_js_parse_int(fa_js_pow(10, t - 3) / 2);
  if (t > 4) return fa_js_parse_int(fa_js_pow(10, t - 2) / 2);
  if (t > 2) return fa_js_parse_int(fa_js_pow(10, t / 3));
  if (t > 1) return fa_js_parse_int(y / 10);
  return 1;
}

__device__ __forceinline__ int gate_update_rec(ScanState& st, double e, double& Tb, int& kb) {
  int flags = 0;
  st.w++;
  if (e > st.y || (st.w > 40 && e > 2 * st.v)) {
    if (e >= st.y) { st.w = 0; st.x = st.y = e; }
    else if (100 * e > st.x) { st.y -= fa_js_parse_int(st.y / 8); st.w = 35; }
    st.v = gate_v_of_y(st.y);
    st.v0 = st.v;
    Tb = st.T; kb = st.k;
    flags = 2;
    if (st.k > 0 && st.T < 30 * st.v * (double)st.k) { flags = 3; st.k = 0; st.T = 0; }
    st.T += st.y;
    st.k += 1;
  } else if (st.v > 10 && 10 * st.v > st.v0 && st.w > 20) {
    st.v -= (double)((unsigned)st.v0 / 20u);
    if (st.v < 10) st.v = 10;
  }
  return flags;
}

__device__ __forceinline__ bool gate_update(ScanState& st, double e) {
  double Tb;
  int kb;
  return gate_update_rec(st, e, Tb, kb) & 1;
}

// C() @B28506
__device__ __forceinline__ void noise_gate(ScanState& st, WarpShared& S, double e, const int lane) {
  if (gate_update(st, e)) seg_reset(st, S, 0, lane);
}

// accumulate_fm @B35952
__device__ __forceinline__ void accumulate_fm(const FaSegmentParams& p, WarpShared& S, ScanState& st, const Bases& bs,
                                              const int n_peaks, const int n_label, const double g, const double vmin,
                                              const int lane) {
  if (n_peaks < 1) return;
  st.s_energy += g;
  const unsigned lt = (1u << lane) - 1u;
  int B = p.B;
  asm volatile("" : "+r"(B));
  const int n_slots = st.n_slots;
  unsigned long long* spill = p.cs_spill + (size_t)bs.spill * ((CMAX - CSM) * ACAP);  // > 3 scoring candidates in a window: rare
  // (1) lane per track slot: expire, window of candidate peaks, scores, arg-max per peak (atomicMax on the bits)
  bool bad = false;
  for (int r0 = 0; r0 < n_slots; r0 += 32) {
    const int r = r0 + lane;
    const int id = S.t_id[r];
    const int gap = n_label - S.t_lf[r];
    unsigned kept = 0u;
    if (id >= 0) {
      if (gap >= 4) S.t_id[r] = -1;  // can never match again (the reference keeps it but never touches it)
      else if (gap >= 0) {
        const int lb = S.t_bins[r] & 255;
        const int lim = gap == 0 ? 3 : gap == 1 ? 4 : gap == 2 ? 6 : 9;  // DIST @B32325
        const int wlo = max(lb - lim + 1, 0), whi = min(lb + lim - 1, B - 1);
        const int word = wlo >> 5, sh = wlo & 31;
        const unsigned long long two = (unsigned long long)S.pmask[word] | ((unsigned long long)S.pmask[word + 1] << 32);
        unsigned bits = (unsigned)(two >> sh) & ((2u << (whi - wlo)) - 1u);
        if (bits) {
          const double amp_old = (double)S.t_amp[r], vel = S.t_vel[r];
          const int np = S.t_np[r];
          int j = 0;
          do {
            const int b = __ffs(bits) - 1;
            bits &= bits - 1;
            const int bin = wlo + b;
            const int o = S.pidx[bin];
            const double sc = fm_score(gap, (double)abs(lb - bin), np, lb, bin, amp_old, (double)S.pa[o].y, vel);
            if (sc > 1) {
              const unsigned long long sb = (unsigned long long)__double_as_longlong(sc);
              if (j < CSM) S.cs[j][r] = sb;
              else if (j < CMAX) spill[(j - CSM) * ACAP + r] = sb;
              j++;
              kept |= 1u << b;
              atomicMax(&S.best[o], sb);
            }
          } while (bits);
          bad |= j > CMAX;
        }
      }
    }
    S.t_wm[r] = kept;
  }
  if (__any_sync(FULL, bad)) { st.overflow = 1; return; }
  __syncwarp();
  // exact ties go to the earlier track
  for (int r0 = 0; r0 < n_slots; r0 += 32) {
    const int r = r0 + lane;
    unsigned bits = S.t_wm[r];
    if (bits) {
      const int id = S.t_id[r];
      const int gap = n_label - S.t_lf[r];
      const int lb = S.t_bins[r] & 255;
      const int lim = gap == 0 ? 3 : gap == 1 ? 4 : gap == 2 ? 6 : 9;
      const int wlo = max(lb - lim + 1, 0);
      int j = 0;
      do {
        const int b = __ffs(bits) - 1;
        bits &= bits - 1;
        const int o = S.pidx[wlo + b];
        const unsigned long long mine = j < CSM ? S.cs[j][r] : spill[(j - CSM) * ACAP + r];
        if (mine == S.best[o]) atomicMin(&S.owner[o], id);
        j++;
      } while (bits);
    }
  }
  __syncwarp();
  // (2) every owning track absorbs its (merged) peaks
  unsigned long long moved = 0;
  for (int r0 = 0; r0 < n_slots; r0 += 32) {
    const int r = r0 + lane;
    unsigned bits = S.t_wm[r];
    uint32_t amp0 = 0, bamp = 0;
    int ob = 0, lo_b = 0, hi_b = 0, id = -1, tb = 0;
    unsigned long long pl = 0, ph = 0;
    if (bits) {
      id = S.t_id[r];
      tb = S.t_bins[r];
      const int gap = n_label - S.t_lf[r];
      const int lb = tb & 255;
      const int lim = gap == 0 ? 3 : gap == 1 ? 4 : gap == 2 ? 6 : 9;
      const int wlo = max(lb - lim + 1, 0);
      do {
        const int b = __ffs(bits) - 1;
        bits &= bits - 1;
        const int bin = wlo + b;
        const int o = S.pidx[bin];
        if (S.owner[o] == id) {
          const uint2 pa = S.pa[o];
          const ulonglong2 e2 = S.plh[o];
          const int l_b = pa.x & 0xff, h_b = (pa.x >> 8) & 0xff;
          if (amp0 == 0u) { amp0 = pa.y; bamp = pa.y; ob = bin; pl = e2.x; ph = e2.y; lo_b = l_b; hi_b = h_b; }
          else {
            pl = e2.x < pl ? e2.x : pl; ph = e2.y > ph ? e2.y : ph; lo_b = min(lo_b, l_b); hi_b = max(hi_b, h_b);
            if (pa.y > bamp) { bamp = pa.y; ob = bin; }
          }
        }
      } while (bits);
    }
    const bool upd = amp0 != 0u && (double)amp0 > vmin;
    const unsigned um = __ballot_sync(FULL, upd);
    if (upd) {
      const unsigned long long Ei = ph - pl;
      const double E = (double)Ei;
      moved += Ei;
      const int h = S.t_np[r];
      const int b1 = tb & 255, b2 = (tb >> 8) & 255, b3 = (tb >> 16) & 255;
      if (h >= 3) S.t_vel[r] = (double)(ob - b1 + (b2 - b1) + (b3 - b2)) / 3;
      else if (h == 2) S.t_vel[r] = (double)(ob - b1 + (b2 - b1)) / 2;
      else if (h == 1) S.t_vel[r] = (double)(ob - b1);
      const double se = S.t_se[r] + E, seb = S.t_seb[r] + E * (double)ob;
      S.t_lf[r] = n_label; S.t_bins[r] = ob | (b1 << 8) | (b2 << 16); S.t_amp[r] = amp0; S.t_np[r] = h + 1;
      S.t_se[r] = se; S.t_seb[r] = seb;
      const long long q = bs.pb + st.n_pts + __popc(um & lt);
      p.pt_track[q] = id; p.pt_ord[q] = h; p.pt_frame[q] = n_label;
      p.pt_binspan[q] = ob | (lo_b << 8) | ((hi_b - lo_b + 1) << 16); p.pt_e[q] = E;
      if (p.pt_amp) p.pt_amp[q] = amp0;
      const long long ti = bs.tb + id;
      p.trk_count[ti] = h + 1; p.trk_sum_e[ti] = se; p.trk_sum_eb[ti] = seb;
    }
    st.n_pts += __popc(um);
  }
  {
    const double mv = (double)warp_sum_u64(moved);  // exact integers: one subtraction == the reference's sequence
    st.s_energy -= mv;
    st.c_energy += mv;
  }
  // (3) un-owned peaks above the gate start new tracks, in peak order, in free slots
  int nn = 0;
  for (int o0 = 0; o0 < n_peaks; o0 += 32) {
    const int o = o0 + lane;
    const bool mk = o < n_peaks && S.owner[o] == BIG && (double)S.pa[o].y > vmin;
    const unsigned nm = __ballot_sync(FULL, mk);
    if (mk) S.newlist[nn + __popc(nm & lt)] = (unsigned char)o;
    nn += __popc(nm);
  }
  if (nn > 0) {
    if (st.n_tr + nn > bs.tcap) { st.overflow = 1; return; }
    __syncwarp();
    int taken = 0, hw = n_slots;
    for (int r0 = 0; r0 < ACAP && taken < nn; r0 += 32) {
      const int r = r0 + lane;
      const bool fr = r >= n_slots || S.t_id[r] < 0;
      const unsigned fm = __ballot_sync(FULL, fr);
      const int i = taken + __popc(fm & lt);
      if (fr && i < nn) {
        const int o = S.newlist[i];
        const uint2 pa = S.pa[o];
        const ulonglong2 e2 = S.plh[o];
        const int pk = (pa.x >> 16) & 0xff;
        const double E = (double)(e2.y - e2.x);
        const int id = st.n_tr + i;
        S.t_id[r] = id; S.t_lf[r] = n_label; S.t_bins[r] = pk; S.t_amp[r] = pa.y; S.t_vel[r] = 0; S.t_np[r] = 1;
        S.t_se[r] = E; S.t_seb[r] = E * (double)pk; S.t_wm[r] = 0u;
        const long long q = bs.pb + st.n_pts + i;
        p.pt_track[q] = id; p.pt_ord[q] = 0; p.pt_frame[q] = n_label;
        p.pt_binspan[q] = pk | ((int)(pa.x & 0xff) << 8) | (((int)((pa.x >> 8) & 0xff) - (int)(pa.x & 0xff) + 1) << 16); p.pt_e[q] = E;
        if (p.pt_amp) p.pt_amp[q] = pa.y;
        const long long ti = bs.tb + id;
        p.trk_count[ti] = 1; p.trk_sum_e[ti] = E; p.trk_sum_eb[ti] = E * (double)pk;
      }
      // new high-water mark: one past the last slot taken in this pass
      const unsigned took = __ballot_sync(FULL, fr && i < nn);
      if (took) hw = max(hw, r0 + 32 - __clz(took));
      taken += __popc(fm);
    }
    if (taken < nn) { st.overflow = 1; return; }
    st.n_slots = hw;
    st.n_tr += nn;
    st.n_pts += nn;
  }
}

// O() @B27088, fast path: the segment's tables (T tracks, len rows, n_pts points) fit the per-frame shared-memory bytes
// that are dead during finalisation.  Same results as finalize_segment below, which works in HBM for any size.
//   scratch: mean f64[T] | rank u8[T] | slot s8[T] | order u8[T] | rc i32[len] | ro i32[len] | key u32[cap]
//   key = rank << 24 | ordinal << 14 | point << 2 | slot  (T <= 255, ordinal < 1024, point < 4096)
//   (Keeping the points' energy / bin / span beside the keys was tried: 12 B per point instead of 4 no longer fits the
//   1000-1600 selected points of a synthetic-speech segment, and more shared memory per warp squeezes the L1 -- so the row
//   pass prefetches its points' pool lines to L1 instead, ahead of the dependent loads.)
// Returns -3 (nothing changed) when the selected points turn out not to fit: the caller then takes the HBM path.
__device__ __forceinline__ bool finalize_fits(const ScanState& st, const int len, const int scratch_bytes) {
  const int T = st.n_tr;
  const int need = ((8 * T + 3 * T + 7) & ~7) + 8 * len;
  return T <= 255 && st.n_pts < 4096 && st.c_ci + 1 < 1024 && len < 1024 && need + 2304 <= scratch_bytes;
}

__device__ __noinline__ int finalize_fast(const FaSegmentParams p, WarpShared& S, ScanState& st, const Bases bs,
                                          const int n_arg, const int lane) {
  const int scratch_bytes = p.smem_per_warp - kScratchOff;
  const int len = n_arg - st.no_fm_segs;
  const int start = st.current_frame - len;
  const double vmin = st.v;
  const int T = st.n_tr, NP = st.n_pts;
  unsigned char* W = reinterpret_cast<unsigned char*>(&S) + kScratchOff;
  double* mean = reinterpret_cast<double*>(W);
  unsigned char* rank = W + 8 * T;
  signed char* slot = reinterpret_cast<signed char*>(rank + T);
  unsigned char* order = rank + 2 * T;
  int* rc = reinterpret_cast<int*>(W + ((11 * T + 7) & ~7));
  int* ro = rc + len;
  unsigned char* tail = W + ((((11 * T + 7) & ~7) + 8 * len + 7) & ~7);
  const int cap_keys = (scratch_bytes - (int)(tail - W)) / 4;
  uint32_t* key = reinterpret_cast<uint32_t*>(tail);
  const unsigned lt = (1u << lane) - 1u;
  __syncwarp();  // the track table is written through at every update (by whichever lane owns the track)
  // get_ranked_formants @B35670: count >= 2, mean >= 7, stable ascending by mean.  Most tracks are one-point noise tracks, so
  // the eligible ones are compacted first (their means and indices, in the not-yet-used key area) and ranked among themselves
  double* cmean = reinterpret_cast<double*>(tail);                  // [nr]   (>= 4 KB are left: finalize_fits)
  unsigned char* cidx = tail + 2048;                                // [nr]
  int nr = 0;
  for (int i0 = 0; i0 < T; i0 += 32) {
    const int i = i0 + lane;
    bool elig = false;
    double m = -1.0;
    if (i < T) {
      m = p.trk_sum_eb[bs.tb + i] / p.trk_sum_e[bs.tb + i];
      elig = p.trk_count[bs.tb + i] >= 2 && m >= 7;
      mean[i] = elig ? m : -1.0;
      slot[i] = -1;
    }
    const unsigned em = __ballot_sync(FULL, elig);
    if (elig) { const int k = nr + __popc(em & lt); cmean[k] = m; cidx[k] = (unsigned char)i; }
    nr += __popc(em);
  }
  for (int r = lane; r < len; r += 32) rc[r] = 0;
  __syncwarp();
  for (int k = lane; k < nr; k += 32) {
    const double m = cmean[k];
    int rk = 0;
#pragma unroll 4
    for (int j = 0; j < nr; j++) {
      const double mj = cmean[j];
      rk += (mj < m || (mj == m && j < k)) ? 1 : 0;   // the compacted list keeps the tracks in creation order
    }
    const int i = cidx[k];
    rank[i] = (unsigned char)rk;
    order[rk] = (unsigned char)i;
  }
  __syncwarp();
  // slot assignment of straighten_formants @B35074 (sequential over the ranking)
  {
    double anchor = 0;
    int sl = 0;
    for (int r = 0; r < nr; r++) {
      const int i = order[r];
      const double m = mean[i];
      if (fabs(m - anchor) > 20) {
        anchor = m;
        sl++;
        if (sl >= 3) break;
      }
      if (lane == 0) slot[i] = (signed char)sl;
    }
  }
  __syncwarp();

  const int si = st.n_segs;
  fa_segment seg;
  seg.start = start; seg.len = len; seg.stored = -1; seg.n_syllables = 0; seg.first_syllable = -1; seg.row_offset = -1;
  seg.ymax = st.y; seg.vmin = st.v; seg.cs_ratio = st.c_energy / st.s_energy;

  // rows: which points land on which frame row.  The pool is appended call by call and the label of a call (the stale
  // c_ci of its frame, quirk #1) grows strictly from the second call of the epoch on, so the points of one row are
  // contiguous in the pool -- except the run at the pool's head (the first call, whose stale label is arbitrary and may
  // name a row that comes again later).  One pass therefore does everything: select (track has a slot), check for the
  // reference's TypeError, compact the selected points' keys and payloads into shared memory in pool order, and note
  // where each row's keys start; the head run is kept as a second key range [0, x_cnt) of row x_row.
  bool thrown = false, nofit = false;
  int n_sel = 0, x_row = -1, x_cnt = 0, last_label = -1;
  {
    const int label0 = NP > 0 ? p.pt_frame[bs.pb] : -1;
    bool in_head = true;
    int tr_n = 0, fr_n = 0, od_n = 0;
    if (lane < NP) { tr_n = p.pt_track[bs.pb + lane]; fr_n = p.pt_frame[bs.pb + lane]; od_n = p.pt_ord[bs.pb + lane]; }
    for (int q0 = 0; q0 < NP; q0 += 32) {
      const int q = q0 + lane;
      const int i = tr_n, fr = fr_n, od = od_n;
      if (q + 32 < NP) {  // next chunk's loads fly while this one is processed
        tr_n = p.pt_track[bs.pb + q + 32]; fr_n = p.pt_frame[bs.pb + q + 32]; od_n = p.pt_ord[bs.pb + q + 32];
      }
      const bool valid = q < NP;
      int head_end = 32;
      if (in_head) {
        const unsigned diff = __ballot_sync(FULL, valid && fr != label0);
        if (diff) { head_end = __ffs(diff) - 1; in_head = false; }
      } else head_end = 0;
      const int sl = valid ? slot[i] : -1;
      bool sel = sl >= 0;
      if (sel && (fr < 0 || fr >= len)) { thrown = true; sel = false; }  // r[d] is undefined -> TypeError -> .catch(L(-1))
      const unsigned sm = __ballot_sync(FULL, sel);
      if (sm) {
        const unsigned before = sm & lt;
        const int pos = n_sel + __popc(before);
        const int prev_lane = before ? 31 - __clz(before) : 0;
        const bool head = lane < head_end;
        const int lab = head ? -1 : fr;   // a head point never continues a row (its row may come again much later)
        int prev_label = __shfl_sync(FULL, lab, prev_lane);
        if (!before) prev_label = last_label;
        if (sel) {
          if (pos >= cap_keys) nofit = true;
          else {
            key[pos] = ((uint32_t)rank[i] << 24) | ((uint32_t)od << 14) | ((uint32_t)q << 2) | (uint32_t)sl;
            if (!head) {
              if (fr != prev_label) ro[fr] = pos;   // first selected point of its row
              atomicAdd(&rc[fr], 1);
            }
          }
        }
        const unsigned hm = sm & (head_end >= 32 ? FULL : (1u << head_end) - 1u);
        if (hm) { x_cnt += __popc(hm); x_row = label0; }
        n_sel += __popc(sm);
        last_label = __shfl_sync(FULL, lab, 31 - __clz(sm));
      }
    }
  }
  thrown = __any_sync(FULL, thrown);
  if (thrown) {
    st.n_segs++;
    if (lane == 0) p.segs[bs.sb + si] = seg;
    return -1;
  }
  if (__any_sync(FULL, nofit)) return -3;  // selected points do not fit: nothing but scratch was touched
  st.n_segs++;
  __syncwarp();
  // apply: lane per row, points ordered by (track rank, point ordinal)
  float* Fout = p.formants + (size_t)(bs.row0 + st.n_rows) * 9;
  float* Eout = p.energy + (size_t)(bs.row0 + st.n_rows) * 3;
  for (int fr = lane; fr < len; fr += 32) {
    const int k1 = rc[fr], off = k1 ? ro[fr] : 0;
    const int k2 = fr == x_row ? x_cnt : 0;   // the head run's keys sit at [0, x_cnt)
    const int k = k1 + k2;
    // the points are visited in (rank, ordinal) order, each visit two dependent loads from the pool: pull the lines to L1 first
    for (int z = 0; z < k; z++) {
      const int q = (int)((key[z < k1 ? off + z : z - k1] >> 2) & 4095u);
      asm volatile("prefetch.global.L1 [%0];" ::"l"(p.pt_e + bs.pb + q));
      asm volatile("prefetch.global.L1 [%0];" ::"l"(p.pt_binspan + bs.pb + q));
    }
    float f0 = 0, f1 = 0, f2 = 0, f3 = 0, f4 = 0, f5 = 0, f6 = 0, f7 = 0, f8 = 0, g0 = 0, g1 = 0, g2 = 0;
    long long last = -1;
    for (int it = 0; it < k; it++) {
      long long bestkey = 0x7fffffffffffffffll;
      for (int z = 0; z < k1; z++) {
        const long long kz = (long long)key[off + z];
        if (kz > last && kz < bestkey) bestkey = kz;
      }
      for (int z = 0; z < k2; z++) {
        const long long kz = (long long)key[z];
        if (kz > last && kz < bestkey) bestkey = kz;
      }
      last = bestkey;
      const int bq = (int)((bestkey >> 2) & 4095);
      int sl = (int)(bestkey & 3);
      const int bs_ = p.pt_binspan[bs.pb + bq];
      const int bin = bs_ & 0xff, span = bs_ >> 16;   // bits 8..15: the point's lower bound (level 3)
      const double E = p.pt_e[bs.pb + bq];
      const float cur = sl == 0 ? f0 : sl == 1 ? f3 : f6;
      if ((double)cur > vmin && (double)cur < (double)bin && sl < 2) sl++;
      const float fb = (float)bin, fe = (float)E, fs = (float)span;
      if (sl == 0) { f0 = fb; f1 = fe; f2 = fs; }
      else if (sl == 1) { f3 = fb; f4 = fe; f5 = fs; }
      else { f6 = fb; f7 = fe; f8 = fs; }
      g0 = (float)((double)g0 + (double)bin * E);
      g1 = (float)((double)g1 + E);
      g2 = (float)((double)g2 + (double)span * E);
    }
    float* fo = Fout + (size_t)fr * 9;
    fo[0] = f0; fo[1] = f1; fo[2] = f2; fo[3] = f3; fo[4] = f4; fo[5] = f5; fo[6] = f6; fo[7] = f7; fo[8] = f8;
    float* eo = Eout + (size_t)fr * 3;
    eo[0] = g0; eo[1] = g1; eo[2] = g2;
    // sep_syllables needs "energy > vmin" per row: keep the flag in rc (row scratch)
    rc[fr] = (double)g1 > vmin ? 1 : 0;
  }
  __syncwarp();
  seg.stored = st.n_stored;
  seg.row_offset = st.n_rows;
  seg.first_syllable = st.n_syls;
  // sep_syllables @B34757
  int nsyl = 0;
  if (p.level == 10 || p.level == 11 || p.level == 12 || p.level == 13) {
    int sstart = -1, quiet = 0, loud = 0;
    for (int e0 = 0; e0 < len; e0 += 32) {
      const int e = e0 + lane;
      const bool is_loud = e < len && rc[e] != 0;
      const unsigned bits = __ballot_sync(FULL, is_loud);
      const int cnt = min(32, len - e0);
      for (int b = 0; b < cnt; b++) {
        const int ee = e0 + b;
        if ((bits >> b) & 1u) { quiet = 0; loud++; if (sstart < 0) sstart = ee; }
        else quiet++;
        if ((loud > 20 && quiet > 0) || (loud > 10 && quiet > 1) || (loud > 0 && quiet > 4) || (ee >= len - 1 && loud > 4)) {
          const int end = ee - quiet;
          if (end - sstart > 1) {
            if (lane == 0) {
              fa_syllable sy;
              sy.stored_seg = st.n_stored; sy.start = sstart; sy.len = end - sstart; sy.reserved = 0;
              p.syls[bs.sb + st.n_syls + nsyl] = sy;
            }
            nsyl++;
            sstart = -1;
            loud = 0;
          }
        }
      }
    }
  }
  seg.n_syllables = nsyl;
  if (lane == 0) p.segs[bs.sb + si] = seg;
  st.n_syls += nsyl;
  st.n_stored++;
  st.n_rows += len;
  __syncwarp();
  return 1;
}

// O() @B27088.  Returns 1 stored, 0 ignored, -1 rejected (where the JS throws inside straighten_formants).
__device__ __noinline__ int finalize_segment(const FaSegmentParams p, ScanState& st, const Bases bs, const int n_arg,
                                             const int lane) {
  const int len = n_arg - st.no_fm_segs;
  if (!(len > p.seg_min_frames && st.c_started >= 2)) return 0;
  const int start = st.current_frame - len;
  const double vmin = st.v;
  __syncwarp();  // the track table is written through at every update (by whichever lane owns the track)
  const int T = st.n_tr;
  // get_ranked_formants @B35670: count >= 2, mean >= 7, stable ascending by mean
  int nr = 0;
  for (int i0 = 0; i0 < T; i0 += 32) {
    const int i = i0 + lane;
    bool elig = false;
    if (i < T) {
      const double m = p.trk_sum_eb[bs.tb + i] / p.trk_sum_e[bs.tb + i];
      elig = p.trk_count[bs.tb + i] >= 2 && m >= 7;
      p.trk_mean[bs.tb + i] = elig ? m : -1.0;
      p.trk_slot[bs.tb + i] = -1;
    }
    nr += __popc(__ballot_sync(FULL, elig));
  }
  __syncwarp();
  for (int i = lane; i < T; i += 32) {
    const double m = p.trk_mean[bs.tb + i];
    if (m >= 7) {
      int rank = 0;
      for (int j = 0; j < T; j++) {
        const double mj = p.trk_mean[bs.tb + j];
        if (mj >= 7 && (mj < m || (mj == m && j < i))) rank++;
      }
      p.trk_rank[bs.tb + i] = rank;
      p.trk_order[bs.tb + rank] = i;
    }
  }
  __syncwarp();
  if (p.level == 3) {
    // O() @B27088, level-3 branch: u.push([e, a]), s.push(get_ranked_formants()), no straighten_formants (nothing can throw).
    // The ranked tracks leave as headers (rank order) + points (time order); tables: base = the utterance's point-pool base.
    const int si3 = st.n_segs;
    fa_track* th = reinterpret_cast<fa_track*>(p.syls) + bs.pb + st.n_syls;
    fa_track_point* tp = p.track_points + bs.pb + st.n_rows;
    int run = 0;
    for (int r0 = 0; r0 < nr; r0 += 32) {
      const int r = r0 + lane;
      const int i = r < nr ? p.trk_order[bs.tb + r] : 0;
      const int c = r < nr ? p.trk_count[bs.tb + i] : 0;
      int incl = c;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(FULL, incl, o);
        if (lane >= o) incl += t;
      }
      if (r < nr) {
        const int off = run + incl - c;
        fa_track h3;
        h3.stored_seg = st.n_stored; h3.first_point = st.n_rows + off; h3.n_points = c; h3.reserved = 0;
        th[r] = h3;
        p.trk_rank[bs.tb + i] = off;      // the rank has done its job: from here on the track's first point
      }
      run += __shfl_sync(FULL, incl, 31);
    }
    __syncwarp();
    for (int q = lane; q < st.n_pts; q += 32) {
      const int i = p.pt_track[bs.pb + q];
      if (p.trk_mean[bs.tb + i] >= 7) {
        const int bs_ = p.pt_binspan[bs.pb + q];
        const int lo_b = (bs_ >> 8) & 0xff;
        fa_track_point o;
        o.frame = p.pt_frame[bs.pb + q]; o.lo = (int16_t)lo_b; o.hi = (int16_t)(lo_b + (bs_ >> 16) - 1); o.bin = (int16_t)(bs_ & 0xff);
        o.reserved = 0; o.amp = (uint32_t)p.pt_amp[bs.pb + q]; o.energy = p.pt_e[bs.pb + q];
        tp[p.trk_rank[bs.tb + i] + p.pt_ord[bs.pb + q]] = o;
      }
    }
    __syncwarp();
    if (lane == 0) {
      fa_segment sg;
      sg.start = start; sg.len = len; sg.stored = st.n_stored; sg.n_syllables = nr; sg.first_syllable = st.n_syls; sg.row_offset = st.n_rows;
      sg.ymax = st.y; sg.vmin = st.v; sg.cs_ratio = st.c_energy / st.s_energy;
      p.segs[bs.sb + si3] = sg;
    }
    st.n_segs++; st.n_stored++; st.n_syls += nr; st.n_rows += run;
    return 1;
  }
  // slot assignment of straighten_formants @B35074 (sequential over the ranking)
  {
    double anchor = 0;
    int slot = 0;
    for (int r = 0; r < nr; r++) {
      const int i = p.trk_order[bs.tb + r];
      const double m = p.trk_mean[bs.tb + i];
      if (fabs(m - anchor) > 20) {
        anchor = m;
        slot++;
        if (slot >= 3) break;
      }
      if (lane == 0) p.trk_slot[bs.tb + i] = (signed char)slot;
    }
  }
  __syncwarp();

  const int si = st.n_segs;
  fa_segment seg;
  seg.start = start; seg.len = len; seg.stored = -1; seg.n_syllables = 0; seg.first_syllable = -1; seg.row_offset = -1;
  seg.ymax = st.y; seg.vmin = st.v; seg.cs_ratio = st.c_energy / st.s_energy;
  st.n_segs++;

  // rows: which points land on which frame row
  int* rc = p.row_count + bs.rb;
  int* ro = p.row_off + bs.rb;
  for (int r = lane; r < len; r += 32) rc[r] = 0;
  __syncwarp();
  bool thrown = false;
  for (int q = lane; q < st.n_pts; q += 32) {
    const int i = p.pt_track[bs.pb + q];
    if (p.trk_slot[bs.tb + i] >= 0) {
      const int fr = p.pt_frame[bs.pb + q];
      if (fr < 0 || fr >= len) thrown = true;  // r[d] is undefined -> TypeError -> .catch(L(-1))
      else atomicAdd(&rc[fr], 1);
    }
  }
  thrown = __any_sync(FULL, thrown);
  if (thrown) {
    if (lane == 0) p.segs[bs.sb + si] = seg;
    return -1;
  }
  __syncwarp();
  {
    int run = 0;
    for (int r0 = 0; r0 < len; r0 += 32) {
      const int r = r0 + lane;
      const int c = r < len ? rc[r] : 0;
      int incl = c;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(FULL, incl, o);
        if (lane >= o) incl += t;
      }
      if (r < len) { ro[r] = run + incl - c; }
      run += __shfl_sync(FULL, incl, 31);
    }
  }
  __syncwarp();
  for (int r = lane; r < len; r += 32) rc[r] = 0;
  __syncwarp();
  for (int q = lane; q < st.n_pts; q += 32) {
    const int i = p.pt_track[bs.pb + q];
    if (p.trk_slot[bs.tb + i] >= 0) {
      const int fr = p.pt_frame[bs.pb + q];
      const int pos = ro[fr] + atomicAdd(&rc[fr], 1);
      p.row_list[bs.pb + pos] = q;
    }
  }
  __syncwarp();
  // apply: lane per row, points ordered by (track rank, point ordinal)
  float* Fout = p.formants + (size_t)(bs.row0 + st.n_rows) * 9;
  float* Eout = p.energy + (size_t)(bs.row0 + st.n_rows) * 3;
  for (int fr = lane; fr < len; fr += 32) {
    const int k = rc[fr], off = ro[fr];
    float f0 = 0, f1 = 0, f2 = 0, f3 = 0, f4 = 0, f5 = 0, f6 = 0, f7 = 0, f8 = 0, g0 = 0, g1 = 0, g2 = 0;
    long long last = -1;
    for (int it = 0; it < k; it++) {
      long long bestkey = 0x7fffffffffffffffll;
      int bq = -1;
      for (int z = 0; z < k; z++) {
        const int q = p.row_list[bs.pb + off + z];
        const int i = p.pt_track[bs.pb + q];
        const long long key = ((long long)p.trk_rank[bs.tb + i] << 32) | (unsigned)p.pt_ord[bs.pb + q];
        if (key > last && key < bestkey) { bestkey = key; bq = q; }
      }
      last = bestkey;
      const int i = p.pt_track[bs.pb + bq];
      int sl = p.trk_slot[bs.tb + i];
      const int bs_ = p.pt_binspan[bs.pb + bq];
      const int bin = bs_ & 0xff, span = bs_ >> 16;   // bits 8..15: the point's lower bound (level 3)
      const double E = p.pt_e[bs.pb + bq];
      const float cur = sl == 0 ? f0 : sl == 1 ? f3 : f6;
      if ((double)cur > vmin && (double)cur < (double)bin && sl < 2) sl++;
      const float fb = (float)bin, fe = (float)E, fs = (float)span;
      if (sl == 0) { f0 = fb; f1 = fe; f2 = fs; }
      else if (sl == 1) { f3 = fb; f4 = fe; f5 = fs; }
      else { f6 = fb; f7 = fe; f8 = fs; }
      g0 = (float)((double)g0 + (double)bin * E);
      g1 = (float)((double)g1 + E);
      g2 = (float)((double)g2 + (double)span * E);
    }
    float* fo = Fout + (size_t)fr * 9;
    fo[0] = f0; fo[1] = f1; fo[2] = f2; fo[3] = f3; fo[4] = f4; fo[5] = f5; fo[6] = f6; fo[7] = f7; fo[8] = f8;
    float* eo = Eout + (size_t)fr * 3;
    eo[0] = g0; eo[1] = g1; eo[2] = g2;
  }
  __syncwarp();
  seg.stored = st.n_stored;
  seg.row_offset = st.n_rows;
  seg.first_syllable = st.n_syls;
  // sep_syllables @B34757
  int nsyl = 0;
  if (p.level == 10 || p.level == 11 || p.level == 12 || p.level == 13) {
    int sstart = -1, quiet = 0, loud = 0;
    for (int e0 = 0; e0 < len; e0 += 32) {
      const int e = e0 + lane;
      const bool is_loud = e < len && (double)Eout[(size_t)e * 3 + 1] > vmin;
      const unsigned bits = __ballot_sync(FULL, is_loud);
      const int cnt = min(32, len - e0);
      for (int b = 0; b < cnt; b++) {
        const int ee = e0 + b;
        if ((bits >> b) & 1u) { quiet = 0; loud++; if (sstart < 0) sstart = ee; }
        else quiet++;
        if ((loud > 20 && quiet > 0) || (loud > 10 && quiet > 1) || (loud > 0 && quiet > 4) || (ee >= len - 1 && loud > 4)) {
          const int end = ee - quiet;
          if (end - sstart > 1) {
            if (lane == 0) {
              fa_syllable sy;
              sy.stored_seg = st.n_stored; sy.start = sstart; sy.len = end - sstart; sy.reserved = 0;
              p.syls[bs.sb + st.n_syls + nsyl] = sy;
            }
            nsyl++;
            sstart = -1;
            loud = 0;
          }
        }
      }
    }
  }
  seg.n_syllables = nsyl;
  if (lane == 0) p.segs[bs.sb + si] = seg;
  st.n_syls += nsyl;
  st.n_stored++;
  st.n_rows += len;
  return 1;
}

// finalisation works on a copy so that the scan state itself stays in registers (the call is out of line)
__device__ __forceinline__ int finalize_copy(const FaSegmentParams& p, WarpShared& S, ScanState& st, const Bases& bs,
                                             const int n_arg, const int lane) {
  const int len = n_arg - st.no_fm_segs;
  if (!(len > p.seg_min_frames && st.c_started >= 2)) return 0;
  ScanState cp = st;
  int r = -3;
  if (p.level != 3 && p.finalize_in_smem && finalize_fits(st, len, p.smem_per_warp - kScratchOff)) {
    r = finalize_fast(p, S, cp, bs, n_arg, lane);
    st.n_slots = ACAP;  // the track slots were used as scratch: the seg_reset that follows clears all of them
  }
  if (r == -3) r = finalize_segment(p, cp, bs, n_arg, lane);
  st.n_segs = cp.n_segs; st.n_stored = cp.n_stored; st.n_rows = cp.n_rows; st.n_syls = cp.n_syls;
  return r;
}

// kBound only sets the register cap (65536 / kBound): 128 -> 127 registers, 640 -> 96, 1024 -> 64
template <int kBound>
__global__ void __launch_bounds__(kBound, 1) fa_segment_kernel(const FaSegmentParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int ui = blockIdx.x * (int)(blockDim.x >> 5) + wib;
  if (ui >= p.utt_count) return;
  const int u = p.utt_begin + ui;
  if (p.redo_only && p.overflow[u] != 2) return;   // second launch behind fa_segment2_kernel: only what it handed back
  WarpShared& S = *reinterpret_cast<WarpShared*>(smem_raw + (size_t)wib * p.smem_per_warp);
  Bases bs;
  bs.row0 = p.frame_off[u];
  bs.F = (int)(p.frame_off[u + 1] - bs.row0);
  bs.tb = p.track_base[u];
  bs.tcap = (int)(p.track_base[u + 1] - bs.tb);
  int maxp = p.maxp;
  bs.pb = bs.row0 * maxp;
  bs.sb = bs.row0 + u;
  bs.rb = bs.sb;
  bs.u = u;
  bs.spill = u;
  const unsigned lt = (1u << lane) - 1u;

  ScanState st;
  st.current_frame = 0; st.no_fm_segs = 0; st.c_ci = 0; st.c_started = -1; st.w = 0; st.k = 0;
  st.y = p.y0; st.v = p.v0; st.x = p.y0; st.v0 = p.v0; st.T = 0; st.s_energy = 0; st.c_energy = 0;
  st.n_tr = 0; st.n_pts = 0; st.n_slots = 0; st.n_segs = 0; st.n_stored = 0; st.n_rows = 0; st.n_syls = 0;
  st.overflow = 0;
  for (int r = lane; r < ACAP; r += 32) S.t_id[r] = -1;
  if (lane <= FA_MAX_BANDS / 32) S.pmask[lane] = 0u;
  __syncwarp();

  // software prefetch of the next frame: count, g, and the first 32 candidates (one per lane)
  uint32_t pkd_next = 0, amp_next = 0;
  unsigned long long pl_next = 0, ph_next = 0;
  int nc_next = 0;
  double g_next = 0;
  auto prefetch = [&](int t) {
    const size_t row = (size_t)(bs.row0 + t);
    nc_next = __ldg(p.ncand + row);
    g_next = __ldg(p.gsum + row);
    if (lane < maxp) {
      const uint4* c4 = reinterpret_cast<const uint4*>(p.cand + row * maxp + lane);
      const uint4 a = __ldg(c4), b = __ldg(c4 + 1);
      pkd_next = a.x; amp_next = a.y; pl_next = a.z | ((unsigned long long)a.w << 32); ph_next = b.x | ((unsigned long long)b.y << 32);
    }
  };
  if (bs.F > 0) prefetch(0);

  for (int t = 0; t < bs.F && !st.overflow; t++) {
    // ---- spectrum_push @B30392 ----
    st.current_frame++;
    const uint32_t pkd0 = pkd_next, amp0 = amp_next;
    const unsigned long long pl0 = pl_next, ph0 = ph_next;
    const int nc = min(nc_next, maxp);
    if (nc_next > maxp) st.overflow = 1;
    const double g = g_next;
    if (t + 1 < bs.F) prefetch(t + 1);

    // ---- D() @B25717: filter the candidates of K2 by the gate v (value at frame start) ----
    const double v = st.v;
    const int t_stale = st.c_ci;
    int n = 0, pbin = 0;
    unsigned long long dsum = 0;
    double h = 2 * v;
    auto filter = [&](const int c0, const uint32_t pkd, const uint32_t amp, const unsigned long long pl,
                      const unsigned long long ph) {
      const bool acc = c0 + lane < nc && (double)amp > v;
      const unsigned m = __ballot_sync(FULL, acc);
      if (m == 0u) return;
      const int pk = (pkd >> 16) & 0xff;
      if (acc) {
        const int pos = n + __popc(m & lt);
        if (pos < PCAP) {
          S.pa[pos] = make_uint2(pkd, amp); S.plh[pos] = make_ulonglong2(pl, ph);
          S.best[pos] = 0ull; S.owner[pos] = BIG;
          S.pidx[pk] = (unsigned char)pos;
          atomicOr(&S.pmask[pk >> 5], 1u << (pk & 31));
        }
      }
      n += __popc(m);
      const uint32_t a = acc ? amp : 0u;
      dsum += (unsigned long long)__reduce_add_sync(FULL, a & 0xffffu) +
              ((unsigned long long)__reduce_add_sync(FULL, a >> 16) << 16);
      // h / p: first strictly greater wins; the last-bin peak never updates them
      const bool hp = acc && !((pkd >> 24) & 1u);
      const uint32_t mx = __reduce_max_sync(FULL, hp ? amp : 0u);
      const unsigned who = __ballot_sync(FULL, hp && amp == mx);
      if (who && (double)mx > h) {
        h = (double)mx;
        pbin = __shfl_sync(FULL, pk, __ffs(who) - 1);
      }
    };
    filter(0, pkd0, amp0, pl0, ph0);
    for (int c0 = 32; c0 < nc; c0 += 32) {  // more than 32 candidates in a frame: rare
      uint4 a = make_uint4(0u, 0u, 0u, 0u), b = a;
      if (c0 + lane < nc) {
        const uint4* c4 = reinterpret_cast<const uint4*>(p.cand + (size_t)(bs.row0 + t) * maxp + c0 + lane);
        a = __ldg(c4); b = __ldg(c4 + 1);
      }
      filter(c0, a.x, a.y, a.z | ((unsigned long long)a.w << 32), b.x | ((unsigned long long)b.y << 32));
    }
    if (n > PCAP) { st.overflow = 1; break; }
    __syncwarp();
    const double d = (double)dsum;
    // exact integer forms of the reference's quotient tests (see gate_update and fa_segctl_kernel)
    const unsigned long long gi = (unsigned long long)g;
    const bool weak = gi > dsum && 10ull * dsum < gi - dsum;       // d / (g - d) < 0.1

    int fin = -2;
    if (st.c_started < 0) {
      bool strong;                                                  // h (n - 1) / (d - h) > 4
      if (p.auto_gate) strong = d > h && h * (double)(n - 1) > 4 * (d - h);
      else strong = (d > h ? h * (double)(n - 1) / (d - h) : 0) > 4;
      if (n > 0 && pbin > 7 && pbin < p.max_voiced_bin && n > 4 && strong) { seg_reset(st, S, 0, lane); st.c_started = 0; }
      else st.no_fm_segs++;
    }
    if (st.c_started >= 0) {
      if (n == 0 || pbin < 7 || pbin >= p.max_voiced_bin || (n > 3 && weak)) {
        st.no_fm_segs++;
        if (st.c_started < 2) st.c_started--;
        else if ((double)st.no_fm_segs >= p.seg_breaker) fin = finalize_copy(p, S, st, bs, st.c_ci + 1, lane);
        else if (p.auto_gate) noise_gate(st, S, h, lane);
      } else {
        if (p.auto_gate) noise_gate(st, S, h, lane);
        accumulate_fm(p, S, st, bs, n, t_stale, g, st.v, lane);
        if (st.c_started < 2) st.c_started++; else st.no_fm_segs = 0;
      }
    }
    st.c_ci++;
    if (fin != -2) seg_reset(st, S, -1, lane);  // the promise's micro-task runs before the next frame
    __syncwarp();
    if (n > 0 && lane <= FA_MAX_BANDS / 32) S.pmask[lane] = 0u;
    __syncwarp();
  }
  // segment_truncate @B30800 (not for the prefix of a stream that is still running: fa_set_truncate)
  if (!st.overflow && !p.no_truncate) {
    finalize_copy(p, S, st, bs, st.c_ci, lane);
    seg_reset(st, S, 1, lane);
  }
  if (lane == 0) {
    p.n_segs[u] = st.n_segs;
    p.n_stored[u] = st.n_stored;
    p.n_rows[u] = st.n_rows;
    p.n_syls[u] = st.n_syls;
    p.overflow[u] = st.overflow;
    // redo behind fa_segment2_kernel + fa_segfin_kernel: the consumers find every utterance's rows through the epoch table,
    // so point it at the dense rows written here
    if (p.epochs)
      for (int si = 0; si < st.n_segs; si++) p.epochs[bs.sb + si].first = p.segs[bs.sb + si].row_offset;
  }
}


// =====================================================================================================================
// K3 v2: the same scan with accumulate_fm restructured for latency (ncu on v1: 40 % of the stall samples were fixed-latency
// dependencies, 17 % shared-memory round trips, 16 % branch resolution -- one warp per utterance has nothing else to issue,
// so the length of the dependent chain per frame IS the run time).  What changes:
//   * ownership is decided in PEAK lanes: phase 1 is one ballot per accepted peak over the track lanes (slot = lane and
//     lane + 32: both register sets in flight at once) and leaves, in the peak's lane, the 64-bit mask of the tracks whose
//     window holds it; phase 2 lets every peak lane score its own claimants (usually one or two) and keep the arg-max with
//     the reference's tie rule (earlier track wins) in registers -- no shared-memory atomics, no second pass for ties;
//   * a track that owns several peaks is a __match_any group of peak lanes: the lowest lane (= first owned peak, the peaks
//     sit in bin order) merges the others by shuffle and updates the track record in place;
//   * new tracks take the i-th free slot straight from the ballots of free lanes (bit select, no list in shared memory);
//   * the velocity quotient k/3 is a two-FMA Markstein step (exact for |k| < 4096: exhaustively checked), k/2 = k * 0.5.
// Limits: 64 live-track slots and 32 accepted peaks per frame.  An utterance / epoch that needs more stops with
// overflow = 2 and is redone by the general kernel above (ACAP 128, PCAP 136) in a second, normally empty launch.
// Same operations on the same operands as accumulate_fm => identical bits (tests: 83 reference-JS vectors, both paths).
// =====================================================================================================================
constexpr int ACAP2 = 64;

// position of the (i + 1)-th set bit of x (i < popc(x))
__device__ __forceinline__ int select64(const unsigned long long x, int i) {
  unsigned w = (unsigned)x;
  int pos = 0;
  const int c = __popc(w);
  if (i >= c) { i -= c; pos = 32; w = (unsigned)(x >> 32); }
  int t = __popc(w & 0xffffu);
  if (i >= t) { i -= t; pos += 16; w >>= 16; }
  t = __popc(w & 0xffu);
  if (i >= t) { i -= t; pos += 8; w >>= 8; }
  t = __popc(w & 0xfu);
  if (i >= t) { i -= t; pos += 4; w >>= 4; }
  t = __popc(w & 0x3u);
  if (i >= t) { i -= t; pos += 2; w >>= 2; }
  if (i >= (int)(w & 1u)) pos += 1;
  return pos;
}

__device__ __forceinline__ unsigned long long shfl_u64(const unsigned long long v, const int src) {
  const unsigned lo = __shfl_sync(FULL, (unsigned)v, src), hi = __shfl_sync(FULL, (unsigned)(v >> 32), src);
  return (unsigned long long)lo | ((unsigned long long)hi << 32);
}

// accumulate_fm @B35952.  m: lanes that hold an accepted peak of this frame (ascending bin order); the peak's packed bounds,
// amplitude and prefix sums are in that lane's registers.
__device__ __forceinline__ void accumulate_fm2(const FaSegmentParams& p, WarpShared& S, ScanState& st, const Bases& bs,
                                               const unsigned m, const uint32_t my_pkd, const uint32_t my_amp,
                                               const unsigned long long my_pl, const unsigned long long my_ph,
                                               const int n_label, const double g, const double vmin, const int lane) {
  if (m == 0u) return;
  st.s_energy += g;
  const unsigned lt = (1u << lane) - 1u;
  const bool useB = st.n_slots > 32;
  // ---- phase 1a, peak lanes: bitmap of the accepted peaks' bins ----
  const bool active = (m >> lane) & 1u;
  const int my_pk = (int)((my_pkd >> 16) & 0xffu);
  if (active) atomicOr(&S.pmask[my_pk >> 5], 1u << (my_pk & 31));
  __syncwarp();
  // ---- phase 0 + 1b, track lanes (slot = lane and lane + 32, both sets in flight): expire; the peaks inside the window
  //      |lastBin - pk| < DIST[gap] (@B32325) are the set bits of the bitmap there; every one is claimed by OR-ing the lane's
  //      bit into the peak's claimant mask wmask[set][bin] (one shared-memory atomic per claim, all claims in parallel) ----
  int idA = S.t_id[lane], idB = -1;
  {
    const int B = p.B;
    auto window = [&](const int slot, int& id, int& wlo) -> unsigned {
      if (id < 0) return 0u;
      const int gap = n_label - S.t_lf[slot];
      if (gap >= 4) { id = -1; S.t_id[slot] = -1; return 0u; }   // can never match again (the reference keeps it, untouched)
      if (gap < 0) return 0u;
      const int lb = S.t_bins[slot] & 255;
      const int lim = (0x9643 >> (4 * gap)) & 15;
      wlo = max(lb - lim + 1, 0);
      const int whi = min(lb + lim - 1, B - 1);
      const int word = wlo >> 5, sh = wlo & 31;
      const unsigned long long two = (unsigned long long)S.pmask[word] | ((unsigned long long)S.pmask[word + 1] << 32);
      return (unsigned)(two >> sh) & ((2u << (whi - wlo)) - 1u);
    };
    int wloA = 0, wloB = 0;
    unsigned bitsA = window(lane, idA, wloA), bitsB = 0u;
    if (useB) { idB = S.t_id[lane + 32]; bitsB = window(lane + 32, idB, wloB); }
    while (bitsA | bitsB) {
      if (bitsA) { const int b = __ffs(bitsA) - 1; bitsA &= bitsA - 1u; atomicOr(&S.wmask[0][wloA + b], 1u << lane); }
      if (bitsB) { const int b = __ffs(bitsB) - 1; bitsB &= bitsB - 1u; atomicOr(&S.wmask[1][wloB + b], 1u << lane); }
    }
  }
  __syncwarp();
  unsigned WA = 0u, WB = 0u;
  if (active) {
    WA = S.wmask[0][my_pk]; S.wmask[0][my_pk] = 0u;
    if (useB) { WB = S.wmask[1][my_pk]; S.wmask[1][my_pk] = 0u; }
  }
  if (lane <= FA_MAX_BANDS / 32) S.pmask[lane] = 0u;
  // ---- phase 2, peak lanes: score the claimants; strict '>' in track order == max score, earliest creation index ----
  unsigned long long best = 0ull;
  int best_id = BIG, best_q = -1, best_np = 0, best_bins = 0;
  while (__any_sync(FULL, (WA | WB) != 0u)) {
    int q = -1;
    if (WA) { q = __ffs(WA) - 1; WA &= WA - 1u; }
    else if (WB) { q = 32 + __ffs(WB) - 1; WB &= WB - 1u; }
    if (q >= 0) {
      const int lf = S.t_lf[q], tb = S.t_bins[q], np = S.t_np[q], id = S.t_id[q];
      const double amp_old = (double)S.t_amp[q], vel = S.t_vel[q];
      const int lb = tb & 255;
      const double sc = fm_score(n_label - lf, (double)abs(lb - my_pk), np, lb, my_pk, amp_old, (double)my_amp, vel);
      if (sc > 1) {
        const unsigned long long sb = (unsigned long long)__double_as_longlong(sc);
        if (sb > best || (sb == best && id < best_id)) { best = sb; best_id = id; best_q = q; best_np = np; best_bins = tb; }
      }
    }
  }
  __syncwarp();   // every claimant record has been read; the owners are rewritten below
  // ---- phase 3: every owning track absorbs its (merged) peaks -- the first owned peak's lane acts for the track ----
  const bool owned = active && best_q >= 0;
  // peak lanes with the same owner: OR the lane bit into the owner slot's word, read it back (MATCH.ANY costs ~450 cycles here)
  if (owned) atomicOr(&S.t_wm[best_q], 1u << lane);
  __syncwarp();
  const unsigned grp = owned ? S.t_wm[best_q] : 0u;
  const bool leader = owned && lane == __ffs(grp) - 1;
  __syncwarp();
  if (leader) S.t_wm[best_q] = 0u;
  int lo_b = (int)(my_pkd & 0xffu), hi_b = (int)((my_pkd >> 8) & 0xffu), ob = my_pk;
  uint32_t bamp = my_amp;
  unsigned long long pl = my_pl, ph = my_ph;
  {
    unsigned rem = leader ? (grp & ~(1u << lane)) : 0u;
    while (__any_sync(FULL, rem != 0u)) {
      const int src = rem ? __ffs(rem) - 1 : lane;
      const uint32_t pkd2 = __shfl_sync(FULL, my_pkd, src), amp2 = __shfl_sync(FULL, my_amp, src);
      const unsigned long long pl2 = shfl_u64(my_pl, src), ph2 = shfl_u64(my_ph, src);
      if (rem) {
        rem &= rem - 1u;
        pl = pl2 < pl ? pl2 : pl; ph = ph2 > ph ? ph2 : ph;
        lo_b = min(lo_b, (int)(pkd2 & 0xffu)); hi_b = max(hi_b, (int)((pkd2 >> 8) & 0xffu));
        if (amp2 > bamp) { bamp = amp2; ob = (int)((pkd2 >> 16) & 0xffu); }   // strict: the first of equal amplitudes stays
      }
    }
  }
  const bool upd = leader && (double)my_amp > vmin;   // the amplitude of the FIRST owned peak decides (and is stored)
  const unsigned um = __ballot_sync(FULL, upd);
  unsigned long long moved = 0ull;
  if (upd) {
    const int q = best_q;
    const unsigned long long Ei = ph - pl;
    const double E = (double)Ei;
    moved = Ei;
    const int h = best_np;
    const int b1 = best_bins & 255, b2 = (best_bins >> 8) & 255, b3 = (best_bins >> 16) & 255;
    if (h >= 3) {
      // k / 3, correctly rounded: q0 = k * fl(1/3), r = k - 3 q0 (exact), q = q0 + r * fl(1/3)   (Markstein; |k| < 4096 checked)
      const double k = (double)(ob - b1 + (b2 - b1) + (b3 - b2)), third = 1.0 / 3.0;
      const double q0 = k * third;
      S.t_vel[q] = fma(fma(-3.0, q0, k), third, q0);
    } else if (h == 2) S.t_vel[q] = (double)(ob - b1 + (b2 - b1)) * 0.5;
    else if (h == 1) S.t_vel[q] = (double)(ob - b1);
    const double se = S.t_se[q] + E, seb = S.t_seb[q] + E * (double)ob;
    S.t_lf[q] = n_label; S.t_bins[q] = ob | (b1 << 8) | (b2 << 16); S.t_amp[q] = my_amp; S.t_np[q] = h + 1;
    S.t_se[q] = se; S.t_seb[q] = seb;
    const long long pq = bs.pb + st.n_pts + __popc(um & lt);
    p.pt_track[pq] = best_id; p.pt_ord[pq] = h; p.pt_frame[pq] = n_label;
    p.pt_binspan[pq] = ob | (lo_b << 8) | ((hi_b - lo_b + 1) << 16); p.pt_e[pq] = E;
    if (p.pt_amp) p.pt_amp[pq] = my_amp;
    const long long ti = bs.tb + best_id;
    p.trk_count[ti] = h + 1; p.trk_sum_e[ti] = se; p.trk_sum_eb[ti] = seb;
  }
  st.n_pts += __popc(um);
  if (um) {
    const double mv = (double)warp_sum_u64(moved);  // exact integers: one subtraction == the reference's sequence
    st.s_energy -= mv;
    st.c_energy += mv;
  }
  // ---- phase 4: un-owned peaks above the gate start new tracks, in peak order, in the free slots ----
  const bool mk = active && best_q < 0 && (double)my_amp > vmin;
  const unsigned nm = __ballot_sync(FULL, mk);
  if (nm) {
    const int nn = __popc(nm);
    if (st.n_tr + nn > bs.tcap) { st.overflow = 1; return; }
    const unsigned fa = __ballot_sync(FULL, idA < 0);
    const unsigned fb = useB ? __ballot_sync(FULL, idB < 0) : FULL;
    const unsigned long long fre = (unsigned long long)fa | ((unsigned long long)fb << 32);
    if (__popcll(fre) < nn) { st.overflow = 2; return; }   // more than 64 live tracks: the general kernel redoes it
    if (mk) {
      const int i = __popc(nm & lt);
      const int q = select64(fre, i);
      const double E = (double)(my_ph - my_pl);
      const int id = st.n_tr + i;
      S.t_id[q] = id; S.t_lf[q] = n_label; S.t_bins[q] = my_pk; S.t_amp[q] = my_amp; S.t_vel[q] = 0; S.t_np[q] = 1;
      S.t_se[q] = E; S.t_seb[q] = E * (double)my_pk;
      const long long pq = bs.pb + st.n_pts + i;
      p.pt_track[pq] = id; p.pt_ord[pq] = 0; p.pt_frame[pq] = n_label;
      p.pt_binspan[pq] = my_pk | ((int)(my_pkd & 0xffu) << 8) | (((int)((my_pkd >> 8) & 0xffu) - (int)(my_pkd & 0xffu) + 1) << 16); p.pt_e[pq] = E;
      if (p.pt_amp) p.pt_amp[pq] = my_amp;
      const long long ti = bs.tb + id;
      p.trk_count[ti] = 1; p.trk_sum_e[ti] = E; p.trk_sum_eb[ti] = E * (double)my_pk;
    }
    st.n_slots = max(st.n_slots, select64(fre, nn - 1) + 1);
    st.n_tr += nn;
    st.n_pts += nn;
  }
  __syncwarp();   // the records written by the peak lanes are read by the track lanes of the next call
}

// one frame's accepted peaks for accumulate_fm2: the candidates of K2 filtered by the gate v, one per lane.  Frames with at
// most 32 candidates (all but noise frames) keep every accepted peak in its candidate's lane; longer candidate lists are
// compacted through shared memory.  Returns false when more than 32 peaks were accepted (-> redo by the general kernel).
struct PeakRegs {
  unsigned m;
  uint32_t pkd, amp;
  unsigned long long pl, ph;
};

// O()'s acceptance test at a finalisation of fa_segment2_kernel; an accepted attempt becomes one FaEpoch record (everything
// finalize_fast / finalize_segment read of the scan state) and one unit of work for fa_segfin_kernel.  The scan itself never
// reads what a finalisation computes: the next frame only needs seg_reset, and the stored / row / syllable counters only place
// outputs, which fa_segfix_kernel numbers afterwards.
__device__ __forceinline__ int finalize_record(const FaSegmentParams& p, ScanState& st, const Bases& bs, const int n_arg,
                                               const int first, const int last, const int lane) {
  const int len = n_arg - st.no_fm_segs;
  if (!(len > p.seg_min_frames && st.c_started >= 2)) return 0;
  if (lane == 0) {
    FaEpoch e;
    e.first = first; e.last = last; e.n_arg = n_arg; e.no_fm_segs = st.no_fm_segs; e.current_frame = st.current_frame;
    e.c_ci = st.c_ci; e.trk_off = first * p.maxp; e.trk_cap = bs.tcap; e.y = st.y; e.v = st.v;
    e.c_energy = st.c_energy; e.s_energy = st.s_energy; e.n_tr = st.n_tr; e.n_pts = st.n_pts;
    p.epochs[bs.sb + st.n_segs] = e;
    const int w = atomicAdd(p.work_count, 1);
    p.work[w] = make_int2(bs.u, st.n_segs);
  }
  st.n_segs++;
  return 1;
}

template <int kBound>
__global__ void __launch_bounds__(kBound, 1) fa_segment2_kernel(const FaSegmentParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int ui = blockIdx.x * (int)(blockDim.x >> 5) + wib;
  if (ui >= p.utt_count) return;
  const int u = p.utt_begin + ui;
  WarpShared& S = *reinterpret_cast<WarpShared*>(smem_raw + (size_t)wib * p.smem_per_warp);
  Bases bs;
  bs.row0 = p.frame_off[u];
  bs.F = (int)(p.frame_off[u + 1] - bs.row0);
  const long long tb0 = p.track_base[u];
  const int tcap0 = (int)(p.track_base[u + 1] - tb0);
  bs.tb = tb0;
  bs.tcap = tcap0;
  int maxp = p.maxp;
  bs.pb = bs.row0 * maxp;
  bs.sb = bs.row0 + u;
  bs.rb = bs.sb;
  bs.u = u;
  bs.spill = u;
  const unsigned lt = (1u << lane) - 1u;
  // Finalisations are recorded (finalize_record) and run by fa_segfin_kernel behind the scan; every epoch then owns the slices
  // of the track table and the point pool that start at its first frame (an epoch of f frames needs at most f * maxp entries
  // of each).  Level 3 (the raw-track export, tables at the utterance's point-pool base) still finalises in the chain.
  const bool defer = p.level != 3;
  int epoch_first = 0;
  auto new_epoch = [&](const int t) {
    if (!defer) return;
    epoch_first = t;
    bs.tb = tb0 + (long long)t * maxp;
    bs.tcap = tcap0 - t * maxp;
    bs.pb = (bs.row0 + t) * maxp;
  };

  ScanState st;
  st.current_frame = 0; st.no_fm_segs = 0; st.c_ci = 0; st.c_started = -1; st.w = 0; st.k = 0;
  st.y = p.y0; st.v = p.v0; st.x = p.y0; st.v0 = p.v0; st.T = 0; st.s_energy = 0; st.c_energy = 0;
  st.n_tr = 0; st.n_pts = 0; st.n_slots = 0; st.n_segs = 0; st.n_stored = 0; st.n_rows = 0; st.n_syls = 0;
  st.overflow = 0;
  for (int r = lane; r < ACAP; r += 32) { S.t_id[r] = -1; S.t_wm[r] = 0u; }
  if (lane <= FA_MAX_BANDS / 32) S.pmask[lane] = 0u;
  for (int r = lane; r < 2 * FA_MAX_BANDS; r += 32) (&S.wmask[0][0])[r] = 0u;
  __syncwarp();

  // software prefetch of the next frame: count, g, and the first 32 candidates (one per lane)
  uint32_t pkd_next = 0, amp_next = 0;
  unsigned long long pl_next = 0, ph_next = 0;
  int nc_next = 0;
  double g_next = 0;
  auto prefetch = [&](int t) {
    const size_t row = (size_t)(bs.row0 + t);
    nc_next = __ldg(p.ncand + row);
    g_next = __ldg(p.gsum + row);
    if (lane < maxp) {
      const uint4* c4 = reinterpret_cast<const uint4*>(p.cand + row * maxp + lane);
      const uint4 a = __ldg(c4), b = __ldg(c4 + 1);
      pkd_next = a.x; amp_next = a.y; pl_next = a.z | ((unsigned long long)a.w << 32); ph_next = b.x | ((unsigned long long)b.y << 32);
    }
  };
  if (bs.F > 0) prefetch(0);

  for (int t = 0; t < bs.F && !st.overflow; t++) {
    // ---- spectrum_push @B30392 ----
    st.current_frame++;
    PeakRegs pr;
    pr.m = 0u; pr.pkd = pkd_next; pr.amp = amp_next; pr.pl = pl_next; pr.ph = ph_next;
    const int nc = min(nc_next, maxp);
    if (nc_next > maxp) st.overflow = 1;
    const double g = g_next;
    if (t + 1 < bs.F) prefetch(t + 1);
    // pauses are short iterations: one frame of look-ahead does not cover a DRAM miss (ncu: 6 % of the stall samples sat on
    // the first use of g) -- pull the candidate rows of frame t + 4 towards L2 now, one 32-byte sector per lane
    if (t + 4 < bs.F && lane < maxp)
      asm volatile("prefetch.global.L2 [%0];" ::"l"(p.cand + (size_t)(bs.row0 + t + 4) * maxp + lane));

    // ---- D() @B25717: filter the candidates of K2 by the gate v (value at frame start) ----
    const double v = st.v;
    const int t_stale = st.c_ci;
    int n = 0, pbin = 0;
    unsigned long long dsum = 0;
    double h = 2 * v;
    const bool one_chunk = nc <= 32;
    auto filter = [&](const int c0, const uint32_t pkd, const uint32_t amp, const unsigned long long pl,
                      const unsigned long long ph) {
      const bool acc = c0 + lane < nc && (double)amp > v;
      const unsigned mm = __ballot_sync(FULL, acc);
      if (mm == 0u) return;
      const int pk = (pkd >> 16) & 0xff;
      if (one_chunk) pr.m = mm;
      else if (acc) {
        const int pos = n + __popc(mm & lt);
        if (pos < 32) { S.pa[pos] = make_uint2(pkd, amp); S.plh[pos] = make_ulonglong2(pl, ph); }
      }
      n += __popc(mm);
      const uint32_t a = acc ? amp : 0u;
      dsum += (unsigned long long)__reduce_add_sync(FULL, a & 0xffffu) +
              ((unsigned long long)__reduce_add_sync(FULL, a >> 16) << 16);
      // h / p: first strictly greater wins; the last-bin peak never updates them
      const bool hp = acc && !((pkd >> 24) & 1u);
      const uint32_t mx = __reduce_max_sync(FULL, hp ? amp : 0u);
      const unsigned who = __ballot_sync(FULL, hp && amp == mx);
      if (who && (double)mx > h) {
        h = (double)mx;
        pbin = __shfl_sync(FULL, pk, __ffs(who) - 1);
      }
    };
    filter(0, pr.pkd, pr.amp, pr.pl, pr.ph);
    for (int c0 = 32; c0 < nc; c0 += 32) {  // more than 32 candidates in a frame: noise frames
      uint4 a = make_uint4(0u, 0u, 0u, 0u), b = a;
      if (c0 + lane < nc) {
        const uint4* c4 = reinterpret_cast<const uint4*>(p.cand + (size_t)(bs.row0 + t) * maxp + c0 + lane);
        a = __ldg(c4); b = __ldg(c4 + 1);
      }
      filter(c0, a.x, a.y, a.z | ((unsigned long long)a.w << 32), b.x | ((unsigned long long)b.y << 32));
    }
    if (n > 32) { st.overflow = 2; break; }   // more accepted peaks than lanes: the general kernel redoes the utterance
    if (!one_chunk) {
      __syncwarp();
      pr.m = n >= 32 ? FULL : ((1u << n) - 1u);
      if (lane < n) {
        const uint2 a = S.pa[lane];
        const ulonglong2 e2 = S.plh[lane];
        pr.pkd = a.x; pr.amp = a.y; pr.pl = e2.x; pr.ph = e2.y;
      }
      __syncwarp();
    }
    const double d = (double)dsum;
    // exact integer forms of the reference's quotient tests (see gate_update and fa_segctl_kernel)
    const unsigned long long gi = (unsigned long long)g;
    const bool weak = gi > dsum && 10ull * dsum < gi - dsum;       // d / (g - d) < 0.1

    int fin = -2;
    if (st.c_started < 0) {
      bool strong;                                                  // h (n - 1) / (d - h) > 4
      if (p.auto_gate) strong = d > h && h * (double)(n - 1) > 4 * (d - h);
      else strong = (d > h ? h * (double)(n - 1) / (d - h) : 0) > 4;
      if (n > 0 && pbin > 7 && pbin < p.max_voiced_bin && n > 4 && strong) {
        seg_reset(st, S, 0, lane); st.c_started = 0; new_epoch(t);
      } else st.no_fm_segs++;
    }
    if (st.c_started >= 0) {
      if (n == 0 || pbin < 7 || pbin >= p.max_voiced_bin || (n > 3 && weak)) {
        st.no_fm_segs++;
        if (st.c_started < 2) st.c_started--;
        else if ((double)st.no_fm_segs >= p.seg_breaker)
          fin = defer ? finalize_record(p, st, bs, st.c_ci + 1, epoch_first, t, lane) : finalize_copy(p, S, st, bs, st.c_ci + 1, lane);
        else if (p.auto_gate && gate_update(st, h)) { seg_reset(st, S, 0, lane); new_epoch(t); }
      } else {
        if (p.auto_gate && gate_update(st, h)) { seg_reset(st, S, 0, lane); new_epoch(t); }
        accumulate_fm2(p, S, st, bs, pr.m, pr.pkd, pr.amp, pr.pl, pr.ph, t_stale, g, st.v, lane);
        if (st.c_started < 2) st.c_started++; else st.no_fm_segs = 0;
      }
    }
    st.c_ci++;
    if (fin != -2) {
      seg_reset(st, S, -1, lane);                  // the promise's micro-task runs before the next frame
      new_epoch(t + 1);
    }
  }
  // segment_truncate @B30800 (not for the prefix of a stream that is still running: fa_set_truncate)
  if (!st.overflow && !p.no_truncate) {
    if (defer) finalize_record(p, st, bs, st.c_ci, epoch_first, bs.F - 1, lane);
    else finalize_copy(p, S, st, bs, st.c_ci, lane);
    seg_reset(st, S, 1, lane);
  }
  if (lane == 0) {
    p.n_segs[u] = st.n_segs;
    p.n_stored[u] = st.n_stored;
    p.n_rows[u] = st.n_rows;
    p.n_syls[u] = st.n_syls;
    p.overflow[u] = st.overflow;
    if (st.overflow == 2 && p.redo_count) atomicAdd(p.redo_count, 1);
  }
}


// =====================================================================================================================
// K3 v3 (impl 3): the serial scan as a two-warp pipeline per utterance -- warp specialisation inside the CTA.
//
// Only the CONTROL part of D() is sequential on its own (candidate filter by the gate, the start / pause tests, the adaptive
// gate): it never reads what accumulate_fm writes (see Mode 1 below).  So one warp (the PRODUCER) runs the control part of every
// frame and hands the tracker one 64-byte record per frame through a ring in shared memory: which clears happen, whether the
// frame reaches accumulate_fm, with which label and thresholds, and the scalars of a finalisation.  The second warp (the
// CONSUMER) only tracks: accept mask from the recorded gate value, accumulate_fm2, finalize_copy, clears -- the same device
// functions as fa_segment2_kernel, called with the same arguments in the same order => the same bits.  The producer runs up to
// kRing frames ahead; the tracker's chain loses the filter's ballots / reductions and the gate's FP64 tests (0.8 of 3.7 us per
// frame on C2), and the kernel has twice the resident warps.
// A CTA = 4 producer warps (warpgroup 0) + 4 consumer warps (warpgroup 1) for 4 utterances; the producers give registers back
// (setmaxnreg.dec) and the consumers take them (setmaxnreg.inc), so that two CTAs stay resident per SM.
// Overflow rules as in fa_segment2_kernel: > 32 accepted peaks in a frame or > 64 live tracks => overflow = 2 => the general
// kernel redoes the utterance in the second launch.
// =====================================================================================================================
constexpr int kRing = 256;                // frames the control warp may run ahead (an utterance of <= 256 frames never blocks it:
                                          // it finishes early and leaves the schedulers to the tracking warps -- with a 32-frame
                                          // ring the producers' wait loop was 28 % of the kernel's instructions)
constexpr int kFins = 80;                 // finalisations in flight: two of them are >= 4 frames apart (2 voiced + 2 pause frames), so
                                          // <= kRing / 4 = 64 lie inside the ring; a slot is reused only after its frame was consumed
constexpr int kPipeUtts = 4;              // utterances per CTA (one producer + one consumer warp each)
constexpr int kPipeRegsProducer = 88, kPipeRegsConsumer = 168;   // 128 * (88 + 168) = the 256 * 128 registers of the launch
constexpr unsigned kRecClearPre = 1u, kRecVoiced = 2u, kRecFin = 4u, kRecClearPost = 8u, kRecEnd = 16u, kRecStop = 32u;

struct __align__(16) PipeRec {
  unsigned flags;        // kRec*; kRecStop: overflow code in bits 8..15
  int label;             // the (possibly stale) frame label accumulate_fm receives
  int nc;                // candidates of the frame (min(count, maxp))
  int fin;               // kRecFin / kRecEnd: slot of the finalisation's scalars
  double v_filter;       // gate at the start of the frame: a candidate is accepted when its amplitude exceeds it
  double vmin;           // gate after C(h): what accumulate_fm receives
};
static_assert(sizeof(PipeRec) == 32, "one record = two 16-byte words");

struct __align__(16) PipeFin {   // what O() @B27088 reads of the control state
  int n_arg, no_fm_segs, current_frame, c_started;
  double y, v;
};

struct PipeShared {
  PipeRec ring[kRing];
  PipeFin fins[kFins];
  volatile int prod;     // records published
  volatile int cons;     // records consumed
  volatile int abort_;   // the consumer gave up (capacity): the producer stops
  int pad;
};

__device__ __forceinline__ void pipe_producer(const FaSegmentParams& p, PipeShared& Q, const int u, const int lane) {
  const long long row0 = p.frame_off[u];
  const int F = (int)(p.frame_off[u + 1] - row0);
  const int maxp = p.maxp;
  ScanState st;
  st.current_frame = 0; st.no_fm_segs = 0; st.c_ci = 0; st.c_started = -1; st.w = 0; st.k = 0;
  st.y = p.y0; st.v = p.v0; st.x = p.y0; st.v0 = p.v0; st.T = 0;
  uint32_t pkd_next = 0, amp_next = 0;
  int nc_next = 0;
  double g_next = 0;
  auto prefetch = [&](int t) {
    const size_t row = (size_t)(row0 + t);
    nc_next = __ldg(p.ncand + row);
    g_next = __ldg(p.gsum + row);
    if (lane < maxp) {
      const uint2 a = __ldg(reinterpret_cast<const uint2*>(p.cand + row * maxp + lane));
      pkd_next = a.x; amp_next = a.y;
    }
  };
  auto ctl_reset = [&](int started) { st.c_ci = 0; st.c_started = started; st.no_fm_segs = 0; };   // L() without clear_fm
  int n_fin = 0;
  auto put_fin = [&](const int n_arg) -> int {   // (a slot is reused only kFins finalisations later: see kFins)
    const int slot = n_fin++ % kFins;
    if (lane == 0) {
      PipeFin f;
      f.n_arg = n_arg; f.no_fm_segs = st.no_fm_segs; f.current_frame = st.current_frame; f.c_started = st.c_started;
      f.y = st.y; f.v = st.v;
      Q.fins[slot] = f;
    }
    return slot;
  };
  auto publish = [&](const int slot_t, const PipeRec& r) -> bool {
    // ring full: the producer is far ahead of the tracker -- sleep instead of spinning (a spinning warp shares its scheduler's
    // issue slots with a tracking warp)
    while (slot_t - Q.cons >= kRing) { if (Q.abort_) return false; __nanosleep(400); }
    if (lane == 0) Q.ring[slot_t % kRing] = r;
    __syncwarp();
    __threadfence_block();
    if (lane == 0) Q.prod = slot_t + 1;
    return true;
  };
  if (F > 0) prefetch(0);
  int t = 0, stop = 0;
  for (; t < F; t++) {
    st.current_frame++;
    const uint32_t pkd0 = pkd_next, amp0 = amp_next;
    const int nc = min(nc_next, maxp);
    if (nc_next > maxp) { stop = 1; break; }
    const double g = g_next;
    if (t + 1 < F) prefetch(t + 1);
    // ---- D() @B25717: filter the candidates of K2 by the gate v (value at frame start) ----
    const double v = st.v;
    PipeRec r;
    r.flags = 0u; r.label = st.c_ci; r.v_filter = v; r.vmin = 0; r.nc = nc; r.fin = 0;
    int n = 0, pbin = 0;
    unsigned long long dsum = 0;
    double h = 2 * v;
    auto filter = [&](const int c0, const uint32_t pkd, const uint32_t amp) {
      const bool acc = c0 + lane < nc && (double)amp > v;
      const unsigned mm = __ballot_sync(FULL, acc);
      if (mm == 0u) return;
      const int pk = (pkd >> 16) & 0xff;
      n += __popc(mm);
      const uint32_t a = acc ? amp : 0u;
      dsum += (unsigned long long)__reduce_add_sync(FULL, a & 0xffffu) +
              ((unsigned long long)__reduce_add_sync(FULL, a >> 16) << 16);
      const bool hp = acc && !((pkd >> 24) & 1u);
      const uint32_t mx = __reduce_max_sync(FULL, hp ? amp : 0u);
      const unsigned who = __ballot_sync(FULL, hp && amp == mx);
      if (who && (double)mx > h) {
        h = (double)mx;
        pbin = __shfl_sync(FULL, pk, __ffs(who) - 1);
      }
    };
    filter(0, pkd0, amp0);
    for (int c0 = 32; c0 < nc; c0 += 32) {
      uint2 a = make_uint2(0u, 0u);
      if (c0 + lane < nc) a = __ldg(reinterpret_cast<const uint2*>(p.cand + (size_t)(row0 + t) * maxp + c0 + lane));
      filter(c0, a.x, a.y);
    }
    if (n > 32) { stop = 2; break; }
    const double d = (double)dsum;
    const unsigned long long gi = (unsigned long long)g;
    const bool weak = gi > dsum && 10ull * dsum < gi - dsum;       // d / (g - d) < 0.1
    if (st.c_started < 0) {
      bool strong;                                                  // h (n - 1) / (d - h) > 4
      if (p.auto_gate) strong = d > h && h * (double)(n - 1) > 4 * (d - h);
      else strong = (d > h ? h * (double)(n - 1) / (d - h) : 0) > 4;
      if (n > 0 && pbin > 7 && pbin < p.max_voiced_bin && n > 4 && strong) { ctl_reset(0); r.flags |= kRecClearPre; }
      else st.no_fm_segs++;
    }
    bool fin = false;
    if (st.c_started >= 0) {
      if (n == 0 || pbin < 7 || pbin >= p.max_voiced_bin || (n > 3 && weak)) {
        st.no_fm_segs++;
        if (st.c_started < 2) st.c_started--;
        else if ((double)st.no_fm_segs >= p.seg_breaker) {
          fin = true;
          r.flags |= kRecFin;
          r.fin = put_fin(st.c_ci + 1);
        } else if (p.auto_gate && gate_update(st, h)) { ctl_reset(0); r.flags |= kRecClearPost; }
      } else {
        if (p.auto_gate && gate_update(st, h)) { ctl_reset(0); r.flags |= kRecClearPre; }
        r.flags |= kRecVoiced;
        r.vmin = st.v;
        if (st.c_started < 2) st.c_started++; else st.no_fm_segs = 0;
      }
    }
    st.c_ci++;
    if (fin) ctl_reset(-1);      // the promise's micro-task runs before the next frame
    if (!publish(t, r)) return;
  }
  PipeRec e;
  e.label = 0; e.nc = 0; e.fin = 0; e.v_filter = 0; e.vmin = 0;
  if (stop) e.flags = kRecStop | ((unsigned)stop << 8);
  else if (p.no_truncate) e.flags = kRecStop;              // prefix of a running stream: no segment_truncate, overflow code 0
  else { e.flags = kRecEnd; e.fin = put_fin(st.c_ci); }   // segment_truncate @B30800
  publish(t, e);
}

__device__ __forceinline__ void pipe_consumer(const FaSegmentParams& p, WarpShared& S, PipeShared& Q, const int u, const int lane) {
  Bases bs;
  bs.row0 = p.frame_off[u];
  bs.F = (int)(p.frame_off[u + 1] - bs.row0);
  bs.tb = p.track_base[u];
  bs.tcap = (int)(p.track_base[u + 1] - bs.tb);
  const int maxp = p.maxp;
  bs.pb = bs.row0 * maxp;
  bs.sb = bs.row0 + u;
  bs.rb = bs.sb;
  bs.u = u;
  bs.spill = u;
  const unsigned lt = (1u << lane) - 1u;
  ScanState st;
  st.current_frame = 0; st.no_fm_segs = 0; st.c_ci = 0; st.c_started = -1; st.w = 0; st.k = 0;
  st.y = p.y0; st.v = p.v0; st.x = p.y0; st.v0 = p.v0; st.T = 0; st.s_energy = 0; st.c_energy = 0;
  st.n_tr = 0; st.n_pts = 0; st.n_slots = 0; st.n_segs = 0; st.n_stored = 0; st.n_rows = 0; st.n_syls = 0;
  st.overflow = 0;
  for (int r = lane; r < ACAP; r += 32) { S.t_id[r] = -1; S.t_wm[r] = 0u; }
  if (lane <= FA_MAX_BANDS / 32) S.pmask[lane] = 0u;
  for (int r = lane; r < 2 * FA_MAX_BANDS; r += 32) (&S.wmask[0][0])[r] = 0u;
  __syncwarp();
  uint32_t pkd_next = 0, amp_next = 0;
  unsigned long long pl_next = 0, ph_next = 0;
  double g_next = 0;
  auto prefetch = [&](int t) {
    const size_t row = (size_t)(bs.row0 + t);
    g_next = __ldg(p.gsum + row);
    if (lane < maxp) {
      const uint4* c4 = reinterpret_cast<const uint4*>(p.cand + row * maxp + lane);
      const uint4 a = __ldg(c4), b = __ldg(c4 + 1);
      pkd_next = a.x; amp_next = a.y; pl_next = a.z | ((unsigned long long)a.w << 32); ph_next = b.x | ((unsigned long long)b.y << 32);
    }
  };
  // clear_fm @B35919 (the tracker's half of L())
  auto clear_tracks = [&]() {
    st.n_tr = 0; st.n_pts = 0; st.s_energy = 0.0; st.c_energy = 0.0;
    for (int r = lane; r < st.n_slots; r += 32) S.t_id[r] = -1;
    st.n_slots = 0;
    __syncwarp();
  };
  auto finalize = [&](const int slot) {
    const PipeFin f = Q.fins[slot];
    st.no_fm_segs = f.no_fm_segs; st.current_frame = f.current_frame; st.c_started = f.c_started; st.y = f.y; st.v = f.v;
    finalize_copy(p, S, st, bs, f.n_arg, lane);
    S.t_wm[lane] = 0u; S.t_wm[lane + 32] = 0u;   // the finalisation used the track slots as scratch
    clear_tracks();
  };
  if (bs.F > 0) prefetch(0);
  for (int t = 0;; t++) {
    while (Q.prod <= t) __nanosleep(40);
    __threadfence_block();
    const PipeRec r = Q.ring[t % kRing];
    if (r.flags & kRecStop) { st.overflow = (int)((r.flags >> 8) & 0xffu); break; }
    if (r.flags & kRecEnd) { finalize(r.fin); break; }
    const uint32_t pkd0 = pkd_next, amp0 = amp_next;
    const unsigned long long pl0 = pl_next, ph0 = ph_next;
    const double g = g_next;
    if (t + 1 < bs.F) prefetch(t + 1);
    if (t + 4 < bs.F && lane < maxp)
      asm volatile("prefetch.global.L2 [%0];" ::"l"(p.cand + (size_t)(bs.row0 + t + 4) * maxp + lane));
    if (r.flags & kRecClearPre) clear_tracks();
    if (r.flags & kRecVoiced) {
      const int nc = r.nc;
      const double v = r.v_filter;
      PeakRegs pr;
      pr.m = 0u; pr.pkd = pkd0; pr.amp = amp0; pr.pl = pl0; pr.ph = ph0;
      if (nc <= 32) {
        pr.m = __ballot_sync(FULL, lane < nc && (double)amp0 > v);
      } else {   // more than 32 candidates (noise frames): the <= 32 accepted ones are compacted through shared memory
        int n = 0;
        for (int c0 = 0; c0 < nc; c0 += 32) {
          uint4 a = make_uint4(pkd0, amp0, (uint32_t)pl0, (uint32_t)(pl0 >> 32)), b = make_uint4((uint32_t)ph0, (uint32_t)(ph0 >> 32), 0u, 0u);
          if (c0 > 0) {
            a = make_uint4(0u, 0u, 0u, 0u); b = a;
            if (c0 + lane < nc) {
              const uint4* c4 = reinterpret_cast<const uint4*>(p.cand + (size_t)(bs.row0 + t) * maxp + c0 + lane);
              a = __ldg(c4); b = __ldg(c4 + 1);
            }
          }
          const bool acc = c0 + lane < nc && (double)a.y > v;
          const unsigned mm = __ballot_sync(FULL, acc);
          if (acc) {
            const int pos = n + __popc(mm & lt);
            if (pos < 32) {
              S.pa[pos] = make_uint2(a.x, a.y);
              S.plh[pos] = make_ulonglong2(a.z | ((unsigned long long)a.w << 32), b.x | ((unsigned long long)b.y << 32));
            }
          }
          n += __popc(mm);
        }
        __syncwarp();
        pr.m = n >= 32 ? FULL : ((1u << n) - 1u);    // n <= 32: the producer stopped the scan otherwise
        if (lane < n) {
          const uint2 a = S.pa[lane];
          const ulonglong2 e2 = S.plh[lane];
          pr.pkd = a.x; pr.amp = a.y; pr.pl = e2.x; pr.ph = e2.y;
        }
        __syncwarp();
      }
      accumulate_fm2(p, S, st, bs, pr.m, pr.pkd, pr.amp, pr.pl, pr.ph, r.label, g, r.vmin, lane);
      if (st.overflow) { Q.abort_ = 1; break; }
    }
    if (r.flags & kRecFin) finalize(r.fin);
    if (r.flags & kRecClearPost) clear_tracks();
    __syncwarp();
    if (lane == 0) Q.cons = t + 1;     // (after the finalisation: its PipeFin slot is free again)
  }
  if (lane == 0) {
    p.n_segs[u] = st.n_segs;
    p.n_stored[u] = st.n_stored;
    p.n_rows[u] = st.n_rows;
    p.n_syls[u] = st.n_syls;
    p.overflow[u] = st.overflow;
    if (st.overflow == 2 && p.redo_count) atomicAdd(p.redo_count, 1);
  }
}

__global__ void __launch_bounds__(2 * kPipeUtts * 32, 2) fa_segment3_kernel(const FaSegmentParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int k = wib & (kPipeUtts - 1);
  const bool consumer = wib >= kPipeUtts;
  const int ui = blockIdx.x * kPipeUtts + k;
  const size_t per_utt = (size_t)p.smem_per_warp + sizeof(PipeShared);
  WarpShared& S = *reinterpret_cast<WarpShared*>(smem_raw + (size_t)k * per_utt);
  PipeShared& Q = *reinterpret_cast<PipeShared*>(smem_raw + (size_t)k * per_utt + p.smem_per_warp);
  if (!consumer && lane == 0) { Q.prod = 0; Q.cons = 0; Q.abort_ = 0; }
  __syncthreads();
  if (consumer) {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(kPipeRegsConsumer));
    if (ui < p.utt_count) pipe_consumer(p, S, Q, p.utt_begin + ui, lane);
  } else {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kPipeRegsProducer));
    if (ui < p.utt_count) pipe_producer(p, Q, p.utt_begin + ui, lane);
  }
}


// =====================================================================================================================
// Mode 1: the scan split in three.  Only the CONTROL state is sequential in time -- the start / pause tests, c_started,
// no_fm_segs, c_ci and the adaptive gate (y, v, ...) depend on the frame's (n, d, h, p, g) and on each other, never on
// the tracks: accumulate_fm has no way back into D() (its only outputs are the track table and the c/s energies read at
// finalisation).  And every finalisation reads tracks that were cleared at a known frame (L(0) / L(-1) / L(1) all end in
// clear_fm).  So:
//   K3a fa_segctl_kernel   warp per utterance, registers only: the control scan.  Per frame it records whether the frame
//                          reaches accumulate_fm, with which (stale) label, and the gate threshold after the frame; per
//                          finalisation attempt that passes O()'s length test it emits one FaEpoch and queues it.
//   K3b fa_segtrack_kernel warp per EPOCH (work queue over the sub-batch): replays the epoch's voiced frames through the
//                          same accumulate_fm and finalises with the recorded scalars.  Segments of one utterance -- and the
//                          541 segments of a one-hour stream -- are tracked in parallel; pauses and abandoned starts cost
//                          nothing here.  Rows / syllables go to provisional places inside the epoch's own frame range.
//   K3c fa_segfix_kernel   warp per utterance: stored indices, dense row / syllable offsets (rows themselves stay put).
// Same arithmetic on the same operands in the same order as the serial kernel => identical bits.
// =====================================================================================================================
constexpr int kCtlWarps = 4;
constexpr unsigned kCtlVoiced = 0x80000000u, kCtlGate = 0x40000000u, kCtlFired = 0x20000000u, kCtlLabel = 0x1fffffffu;

__device__ __forceinline__ void ctl_init(const FaSegmentParams& p, ScanState& st) {
  st.current_frame = 0; st.no_fm_segs = 0; st.c_ci = 0; st.c_started = -1; st.w = 0; st.k = 0;
  st.y = p.y0; st.v = p.v0; st.x = p.y0; st.v0 = p.v0; st.T = 0; st.s_energy = 0; st.c_energy = 0;
  st.n_tr = 0; st.n_pts = 0; st.n_slots = 0; st.n_segs = 0; st.n_stored = 0; st.n_rows = 0; st.n_syls = 0;
  st.overflow = 0;
}

__device__ __forceinline__ void ctl_save(const ScanState& st, const int epoch_first, const int fired, const int n_events,
                                         FaCtlState& o) {
  o.c_started = st.c_started; o.no_fm_segs = st.no_fm_segs; o.c_ci = st.c_ci; o.w = st.w; o.k = st.k; o.epoch_first = epoch_first;
  o.n_epochs = st.n_segs; o.fired = fired; o.overflow = st.overflow; o.n_events = n_events;
  o.y = st.y; o.v = st.v; o.x = st.x; o.v0 = st.v0; o.T = st.T;
}

__device__ __forceinline__ void ctl_load(const FaCtlState& o, ScanState& st, int& epoch_first) {
  st.c_started = o.c_started; st.no_fm_segs = o.no_fm_segs; st.c_ci = o.c_ci; st.w = o.w; st.k = o.k; epoch_first = o.epoch_first;
  st.y = o.y; st.v = o.v; st.x = o.x; st.v0 = o.v0; st.T = o.T;
}

// O()'s acceptance test at a finalisation; an accepted attempt is written to epochs[slot] (slot = seg_ci index, or a
// provisional place while the chunk is speculative) and, when `queue`, becomes one unit of work for K3b
__device__ __forceinline__ void ctl_attempt(const FaSegmentParams& p, ScanState& st, const int epoch_first, const int n_arg,
                                            const int last, const int maxp, const long long slot_base, const int u,
                                            const bool emit, const bool queue, const int lane) {
  const int len = n_arg - st.no_fm_segs;
  if (!(len > p.seg_min_frames && st.c_started >= 2)) return;
  if (emit && lane == 0) {
    FaEpoch e;
    e.first = epoch_first; e.last = last; e.n_arg = n_arg; e.no_fm_segs = st.no_fm_segs;
    // tracks <= points <= accepted peaks <= maxp per frame: the epoch's frame range of the track table always suffices
    e.current_frame = st.current_frame; e.c_ci = st.c_ci; e.trk_off = epoch_first * maxp; e.trk_cap = (last - epoch_first + 1) * maxp;
    e.y = st.y; e.v = st.v;
    p.epochs[slot_base + st.n_segs] = e;
    if (queue) {
      const int w = atomicAdd(p.work_count, 1);
      p.work[w] = make_int2(u, st.n_segs);
    }
  }
  if (emit) st.n_segs++;
}

// frames [t_begin, t_end) of the control scan of utterance u.  outputs: write the per-frame control record (and the T / k
// record of the gate's test when `record`); emit / queue: see ctl_attempt; fired: set when the gate's T/k reset fires.
__device__ __forceinline__ void segctl_range(const FaSegmentParams& p, const int u, const long long row0, const int t_begin,
                                             const int t_end, ScanState& st, int& epoch_first, int& fired, int& n_events,
                                             const bool outputs, const bool record, const long long slot_base, const bool queue,
                                             const int maxp, const int lane) {
  // The frame inputs (count, g, first 32 candidates) are fetched kGroup frames at a time, one group ahead
  constexpr int kGroup = 4;
  uint32_t pkd_n[kGroup], amp_n[kGroup];
  int nc_n[kGroup];
  double g_n[kGroup];
  auto prefetch_group = [&](const int t0) {
#pragma unroll
    for (int k = 0; k < kGroup; k++) {
      const int t = t0 + k;
      pkd_n[k] = 0u; amp_n[k] = 0u; nc_n[k] = 0; g_n[k] = 0.0;
      if (t < t_end) {
        const size_t row = (size_t)(row0 + t);
        nc_n[k] = __ldg(p.ncand + row);
        g_n[k] = __ldg(p.gsum + row);
        if (lane < maxp) {
          const uint2 a = __ldg(reinterpret_cast<const uint2*>(p.cand + row * maxp + lane));
          pkd_n[k] = a.x; amp_n[k] = a.y;
        }
      }
    }
  };
  prefetch_group(t_begin);
  for (int t0 = t_begin; t0 < t_end && !st.overflow; t0 += kGroup) {
   uint32_t pkd_c[kGroup], amp_c[kGroup];
   int nc_c[kGroup];
   double g_c[kGroup];
#pragma unroll
   for (int k = 0; k < kGroup; k++) { pkd_c[k] = pkd_n[k]; amp_c[k] = amp_n[k]; nc_c[k] = nc_n[k]; g_c[k] = g_n[k]; }
   prefetch_group(t0 + kGroup);
#pragma unroll
   for (int k = 0; k < kGroup; k++) {
    const int t = t0 + k;
    if (t >= t_end || st.overflow) break;
    st.current_frame = t + 1;
    const uint32_t pkd0 = pkd_c[k], amp0 = amp_c[k];
    const int nc = min(nc_c[k], maxp);
    if (nc_c[k] > maxp) st.overflow = 1;
    const double g = g_c[k];
    const double v = st.v;
    const int t_stale = st.c_ci;
    int n = 0, pbin = 0;
    unsigned long long dsum = 0;
    double h = 2 * v;
    auto filter = [&](const int c0, const uint32_t pkd, const uint32_t amp) {
      const bool acc = c0 + lane < nc && (double)amp > v;
      const unsigned m = __ballot_sync(FULL, acc);
      if (m == 0u) return;
      const int pk = (pkd >> 16) & 0xff;
      n += __popc(m);
      const uint32_t a = acc ? amp : 0u;
      dsum += (unsigned long long)__reduce_add_sync(FULL, a & 0xffffu) +
              ((unsigned long long)__reduce_add_sync(FULL, a >> 16) << 16);
      const bool hp = acc && !((pkd >> 24) & 1u);
      const uint32_t mx = __reduce_max_sync(FULL, hp ? amp : 0u);
      const unsigned who = __ballot_sync(FULL, hp && amp == mx);
      if (who && (double)mx > h) {
        h = (double)mx;
        pbin = __shfl_sync(FULL, pk, __ffs(who) - 1);
      }
    };
    filter(0, pkd0, amp0);
    for (int c0 = 32; c0 < nc; c0 += 32) {
      uint2 a = make_uint2(0u, 0u);
      if (c0 + lane < nc) a = __ldg(reinterpret_cast<const uint2*>(p.cand + (size_t)(row0 + t) * maxp + c0 + lane));
      filter(c0, a.x, a.y);
    }
    if (n > PCAP) { st.overflow = 1; break; }
    const double d = (double)dsum;
    // d and g are exact integers (sums of uint32): d/(g-d) < 0.1 <=> 10 d < g - d, and with the automatic gate h is an
    // integer too: h (n-1)/(d-h) > 4 <=> h (n-1) > 4 (d-h)   (same argument as in gate_update; d/0 = inf fails both ways)
    const unsigned long long gi = (unsigned long long)g;
    const bool weak = gi > dsum && 10ull * dsum < gi - dsum;
    bool voiced = false, finalised = false;
    int gflags = 0, kb = 0;
    double Tb = 0;
    auto clear = [&](const int started) {   // L(started): the tracks are cleared, a new epoch starts with this frame
      st.c_ci = 0; st.c_started = started; st.no_fm_segs = 0;
      epoch_first = t;
    };
    if (st.c_started < 0) {
      bool strong;
      if (p.auto_gate) strong = d > h && h * (double)(n - 1) > 4 * (d - h);
      else strong = (d > h ? h * (double)(n - 1) / (d - h) : 0) > 4;   // fixed gate: h = 2 v need not be an integer
      if (n > 0 && pbin > 7 && pbin < p.max_voiced_bin && n > 4 && strong) clear(0);
      else st.no_fm_segs++;
    }
    if (st.c_started >= 0) {
      if (n == 0 || pbin < 7 || pbin >= p.max_voiced_bin || (n > 3 && weak)) {
        st.no_fm_segs++;
        if (st.c_started < 2) st.c_started--;
        else if ((double)st.no_fm_segs >= p.seg_breaker) {
          ctl_attempt(p, st, epoch_first, st.c_ci + 1, t, maxp, slot_base, u, outputs, queue, lane);
          finalised = true;
        } else if (p.auto_gate) { gflags = gate_update_rec(st, h, Tb, kb); if (gflags & 1) clear(0); }
      } else {
        if (p.auto_gate) { gflags = gate_update_rec(st, h, Tb, kb); if (gflags & 1) clear(0); }
        voiced = true;
        if (st.c_started < 2) st.c_started++; else st.no_fm_segs = 0;
      }
    }
    st.c_ci++;
    if (finalised) { st.c_ci = 0; st.c_started = -1; st.no_fm_segs = 0; epoch_first = t + 1; }
    if (gflags & 1) fired = 1;
    if (outputs && lane == 0) {
      p.fr_ctl[row0 + t] = (voiced ? (kCtlVoiced | ((unsigned)t_stale & kCtlLabel)) : 0u) | ((gflags & 2) ? kCtlGate : 0u) |
                           ((gflags & 1) ? kCtlFired : 0u);
      p.fr_v[row0 + t] = st.v;
      if (record && (gflags & 2)) {      // the chunk's next reset-test record
        const long long ei = row0 + t_begin + n_events;
        p.fr_T[ei] = Tb; p.fr_k[ei] = kb | ((gflags & 1) ? (int)0x80000000 : 0); p.fr_thr[ei] = 30 * st.v;
      }
    }
    if (record && (gflags & 2)) n_events++;
   }
  }
}

// utterance mode of the control scan: one warp, all frames
__global__ void __launch_bounds__(kCtlWarps * 32) fa_segctl_kernel(const FaSegmentParams p) {
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int ui = blockIdx.x * kCtlWarps + wib;
  if (ui >= p.utt_count) return;
  const int u = p.utt_begin + ui;
  const long long row0 = p.frame_off[u], sb = row0 + u;
  const int F = (int)(p.frame_off[u + 1] - row0);
  int maxp = p.maxp;
  ScanState st;
  ctl_init(p, st);
  int epoch_first = 0, fired = 0;
  int n_events = 0;
  segctl_range(p, u, row0, 0, F, st, epoch_first, fired, n_events, true, false, sb, true, maxp, lane);
  st.current_frame = F;
  if (!st.overflow && !p.no_truncate) ctl_attempt(p, st, epoch_first, st.c_ci, F - 1, maxp, sb, u, true, true, lane);   // segment_truncate @B30800
  if (lane == 0) {
    p.n_segs[u] = st.n_segs;
    p.overflow[u] = st.overflow;
  }
}

// stream mode, pass 1: warp per chunk.  Chunk 0 starts from the initial state (exact); chunk j > 0 warms up over the
// ctl_warm frames in front of it (no outputs), notes the state it arrives with (its SPECULATED entry) and scans its frames
// with all outputs; accepted finalisations go to provisional slots at the chunk's own first frame.
__global__ void __launch_bounds__(kCtlWarps * 32) fa_segctl_chunk_kernel(const FaSegmentParams p) {
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int wi = blockIdx.x * kCtlWarps + wib;
  if (wi >= p.n_cchunks) return;
  const int u = p.cchunk_utt[wi], j = p.cchunk_idx[wi];
  const long long row0 = p.frame_off[u], sb = row0 + u;
  const int F = (int)(p.frame_off[u + 1] - row0);
  int maxp = p.maxp;
  const int a = j * p.ctl_chunk, b = min(F, a + p.ctl_chunk);
  const long long slot = p.cchunk_base[u] + j;
  ScanState st;
  ctl_init(p, st);
  int epoch_first = 0, fired = 0;
  if (j > 0) {
    int none = 0;
    segctl_range(p, u, row0, max(0, a - p.ctl_warm), a, st, epoch_first, fired, none, false, false, 0, false, maxp, lane);
    st.n_segs = 0;
    fired = 0;
    if (lane == 0) ctl_save(st, epoch_first, 0, 0, p.ctl_entry[slot]);
  }
  int n_events = 0;
  segctl_range(p, u, row0, a, b, st, epoch_first, fired, n_events, true, true, sb + a, false, maxp, lane);
  if (lane == 0) ctl_save(st, epoch_first, fired, n_events, p.ctl_exit[slot]);
}

// stream mode, pass 2: warp per utterance walks the chain of chunks.
__global__ void __launch_bounds__(kCtlWarps * 32) fa_segctl_verify_kernel(const FaSegmentParams p) {
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int ui = blockIdx.x * kCtlWarps + wib;
  if (ui >= p.utt_count) return;
  const int u = p.utt_begin + ui;
  const long long row0 = p.frame_off[u], sb = row0 + u;
  const int F = (int)(p.frame_off[u + 1] - row0);
  int maxp = p.maxp;
  const int nc = (int)(p.cchunk_base[u + 1] - p.cchunk_base[u]);
  ScanState st;          // the TRUE state at the current chunk boundary
  ctl_init(p, st);
  int epoch_first = 0, n_segs = 0, overflow = 0;
  for (int j = 0; j < nc && !overflow; j++) {
    const int a = j * p.ctl_chunk, b = min(F, a + p.ctl_chunk);
    const long long slot = p.cchunk_base[u] + j;
    const FaCtlState X = p.ctl_exit[slot];
    bool ok = true;
    double dT = 0;
    int dk = 0;
    if (j > 0) {
      const FaCtlState G = p.ctl_entry[slot];
      ok = G.c_started == st.c_started && G.no_fm_segs == st.no_fm_segs && G.c_ci == st.c_ci && G.w == st.w &&
           G.epoch_first == epoch_first && G.y == st.y && G.v == st.v && G.x == st.x && G.v0 == st.v0;
      dT = st.T - G.T;
      dk = st.k - G.k;
      if (ok && (dT != 0 || dk != 0)) {
        // T and k are running sums since the gate's last reset: the speculated ones differ from the true ones by a constant
        // until the first reset inside the chunk.  Replay the reset test of every frame up to (and including) that one with
        // the true sums; the chunk stands iff every outcome is what the speculative scan saw.
        const long long e0 = row0 + a;
        int first = 0x7fffffff;
        for (int i = lane; i < X.n_events; i += 32)
          if (p.fr_k[e0 + i] < 0) { first = i; break; }
        first = __reduce_min_sync(FULL, first);
        bool bad = false;
        for (int i = lane; i < X.n_events && i <= first; i += 32) {
          const int kr = p.fr_k[e0 + i];
          const double Tt = p.fr_T[e0 + i] + dT;
          const int kt = (kr & 0x7fffffff) + dk;
          const bool fire = kt > 0 && Tt < p.fr_thr[e0 + i] * (double)kt;
          bad |= fire != (kr < 0);
        }
        ok = !__any_sync(FULL, bad);
      }
    }
    if (ok) {
      // accept: move the chunk's finalisations from their provisional slots (at frame a) to their seg_ci indices and queue them
      if (a != n_segs)
        for (int i = 0; i < X.n_epochs; i++) {       // ascending, dst <= src: in place
          FaEpoch e;
          if (lane == 0) { e = p.epochs[sb + a + i]; p.epochs[sb + n_segs + i] = e; }
        }
      if (lane == 0)
        for (int i = 0; i < X.n_epochs; i++) {
          const int w = atomicAdd(p.work_count, 1);
          p.work[w] = make_int2(u, n_segs + i);
        }
      n_segs += X.n_epochs;
      ctl_load(X, st, epoch_first);
      if (!X.fired) { st.T = X.T + dT; st.k = X.k + dk; }
      overflow |= X.overflow;
    } else {
      // the warm-up had not reached the true state: rescan the chunk from it
      if (lane == 0) atomicAdd(p.ctl_fixups, 1);
      int fired = 0;
      st.n_segs = n_segs;
      st.overflow = 0;
      int none = 0;
      segctl_range(p, u, row0, a, b, st, epoch_first, fired, none, true, false, sb, true, maxp, lane);
      n_segs = st.n_segs;
      overflow |= st.overflow;
    }
    __syncwarp();
  }
  st.n_segs = n_segs;
  st.current_frame = F;
  st.overflow = overflow;
  if (!overflow && !p.no_truncate) ctl_attempt(p, st, epoch_first, st.c_ci, F - 1, maxp, sb, u, true, true, lane);   // segment_truncate @B30800
  if (lane == 0) {
    p.n_segs[u] = st.n_segs;
    p.overflow[u] = overflow;
  }
}

template <int kBound>
__global__ void __launch_bounds__(kBound, 1) fa_segtrack_kernel(const FaSegmentParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  WarpShared& S = *reinterpret_cast<WarpShared*>(smem_raw + (size_t)wib * p.smem_per_warp);
  const int worker = blockIdx.x * (int)(blockDim.x >> 5) + wib;
  int maxp = p.maxp;
  const unsigned lt = (1u << lane) - 1u;
  const int n_work = *reinterpret_cast<volatile int*>(p.work_count);
  for (;;) {
    int wi = 0;
    if (lane == 0) wi = atomicAdd(p.work_count + 1, 1);
    wi = __shfl_sync(FULL, wi, 0);
    if (wi >= n_work) break;
    const int2 wk = p.work[wi];
    const int u = wk.x;
    Bases bs;
    bs.row0 = p.frame_off[u];
    bs.F = (int)(p.frame_off[u + 1] - bs.row0);
    bs.sb = bs.row0 + u;
    const FaEpoch E = p.epochs[bs.sb + wk.y];
    bs.tb = p.track_base[u] + E.trk_off;
    bs.tcap = E.trk_cap;
    bs.pb = (bs.row0 + E.first) * maxp;     // the epoch's own frame range of the point pool
    bs.rb = bs.sb + E.first;                // ... and of the row scratch
    bs.u = u;
    bs.spill = worker;
    ScanState st;
    // pass 0: tracking with peak-lane ownership (accumulate_fm2: <= 64 live tracks, <= 32 accepted peaks per frame); an epoch
    // that needs more (overflow == 2) is replayed by pass 1, the general accumulate_fm -- same rule as the serial kernels
    for (int pass = p.impl == 1 ? 1 : 0; pass < 2; pass++) {
      const bool fast = pass == 0;
      st.current_frame = E.current_frame; st.no_fm_segs = E.no_fm_segs; st.c_ci = E.c_ci; st.c_started = 2;
      st.w = 0; st.k = 0; st.y = E.y; st.v = E.v; st.x = E.y; st.v0 = E.v; st.T = 0; st.s_energy = 0; st.c_energy = 0;
      st.n_tr = 0; st.n_pts = 0; st.n_slots = 0;
      st.n_segs = wk.y;         // -> segs[sb + seg_ci index]
      st.n_stored = 0;          // provisional: K3c numbers the stores
      st.n_rows = E.first;      // provisional row offset: rows land inside the epoch's frame range (len <= its frames)
      st.n_syls = E.first;      // provisional syllable offset, same argument
      st.overflow = 0;
      for (int r = lane; r < ACAP; r += 32) { S.t_id[r] = -1; S.t_wm[r] = 0u; }
      if (lane <= FA_MAX_BANDS / 32) S.pmask[lane] = 0u;
      for (int r = lane; r < 2 * FA_MAX_BANDS; r += 32) (&S.wmask[0][0])[r] = 0u;
      __syncwarp();
      // software prefetch of the next frame's control record, thresholds, count, g and first 32 candidates
      unsigned ctl_n = 0u;
      double v_n = 0, vmin_n = 0, g_n = 0;
      int nc_n = 0;
      uint4 a_n = make_uint4(0u, 0u, 0u, 0u), b_n = a_n;
      auto prefetch = [&](const int t) {
        const size_t row = (size_t)(bs.row0 + t);
        ctl_n = __ldg(p.fr_ctl + row);
        v_n = t > 0 ? __ldg(p.fr_v + row - 1) : p.v0;   // the gate at the start of the frame
        vmin_n = __ldg(p.fr_v + row);                   // ... and after C(h): what accumulate_fm receives
        nc_n = __ldg(p.ncand + row);
        g_n = __ldg(p.gsum + row);
        if (lane < maxp) {
          const uint4* c4 = reinterpret_cast<const uint4*>(p.cand + row * maxp + lane);
          a_n = __ldg(c4); b_n = __ldg(c4 + 1);
        }
      };
      if (E.first <= E.last) prefetch(E.first);
      for (int t = E.first; t <= E.last && !st.overflow; t++) {
        const size_t row = (size_t)(bs.row0 + t);
        const unsigned ctl = ctl_n;
        const double v = v_n, vmin = vmin_n, g = g_n;
        const int nc = min(nc_n, maxp);
        const uint4 a0 = a_n, b0 = b_n;
        if (t < E.last) prefetch(t + 1);
        if (!(ctl >> 31)) continue;
        int n = 0;
        PeakRegs pr;
        pr.m = 0u; pr.pkd = a0.x; pr.amp = a0.y; pr.pl = a0.z | ((unsigned long long)a0.w << 32); pr.ph = b0.x | ((unsigned long long)b0.y << 32);
        if (fast && nc <= 32) {
          pr.m = __ballot_sync(FULL, lane < nc && (double)a0.y > v);
          n = __popc(pr.m);
        } else {
          for (int c0 = 0; c0 < nc; c0 += 32) {
            uint4 a = a0, b = b0;
            if (c0 > 0) {
              a = make_uint4(0u, 0u, 0u, 0u); b = a;
              if (c0 + lane < nc) {
                const uint4* c4 = reinterpret_cast<const uint4*>(p.cand + row * maxp + c0 + lane);
                a = __ldg(c4); b = __ldg(c4 + 1);
              }
            }
            const uint32_t pkd = a.x, amp = a.y;
            const bool acc = c0 + lane < nc && (double)amp > v;
            const unsigned m = __ballot_sync(FULL, acc);
            if (m == 0u) continue;
            if (acc) {
              const int pk = (pkd >> 16) & 0xff;
              const int pos = n + __popc(m & lt);
              if (pos < (fast ? 32 : PCAP)) {
                S.pa[pos] = make_uint2(pkd, amp);
                S.plh[pos] = make_ulonglong2(a.z | ((unsigned long long)a.w << 32), b.x | ((unsigned long long)b.y << 32));
                if (!fast) {
                  S.best[pos] = 0ull; S.owner[pos] = BIG;
                  S.pidx[pk] = (unsigned char)pos;
                  atomicOr(&S.pmask[pk >> 5], 1u << (pk & 31));
                }
              }
            }
            n += __popc(m);
          }
          if (fast) {
            if (n > 32) { st.overflow = 2; break; }
            __syncwarp();
            pr.m = n >= 32 ? FULL : ((1u << n) - 1u);
            if (lane < n) {
              const uint2 a = S.pa[lane];
              const ulonglong2 e2 = S.plh[lane];
              pr.pkd = a.x; pr.amp = a.y; pr.pl = e2.x; pr.ph = e2.y;
            }
          }
        }
        if (n > PCAP) { st.overflow = 1; break; }
        __syncwarp();
        if (fast) {
          accumulate_fm2(p, S, st, bs, pr.m, pr.pkd, pr.amp, pr.pl, pr.ph, (int)(ctl & kCtlLabel), g, vmin, lane);
        } else {
          accumulate_fm(p, S, st, bs, n, (int)(ctl & kCtlLabel), g, vmin, lane);
          __syncwarp();
          if (lane <= FA_MAX_BANDS / 32) S.pmask[lane] = 0u;
        }
        __syncwarp();
      }
      if (fast && st.overflow == 2) {   // hand the epoch to the general path
        if (lane == 0 && p.redo_count) atomicAdd(p.redo_count, 1);
        continue;
      }
      break;
    }
    if (!st.overflow) {
      const int len = E.n_arg - st.no_fm_segs;
      int r = -3;
      if (p.finalize_in_smem && finalize_fits(st, len, p.smem_per_warp - kScratchOff)) r = finalize_fast(p, S, st, bs, E.n_arg, lane);
      if (r == -3) r = finalize_segment(p, st, bs, E.n_arg, lane);
    }
    if (st.overflow && lane == 0) p.overflow[u] = 1;
    __syncwarp();
  }
}

// =====================================================================================================================
// The finaliser of the utterance-mode scan: O() @B27088 for every FaEpoch record fa_segment2_kernel wrote, one CTA per
// record (a persistent grid pulls them from the work list).  Every thread takes part in staging and ranking the eligible
// tracks, counting the selected points per row and scattering their sort keys and payloads (bin / span, energy) into shared
// memory, row by row; after that the record needs no global load: the apply runs one thread per row, the syllable scan one
// warp.  Only the SELECTED points are staged (most tracks are one-point noise tracks that get no slot), 20 B each.  The
// arithmetic and its order are finalize_fast's: count-smaller ranking with the creation-order tie rule, the sequential slot
// rule of straighten_formants, visits in (rank, ordinal) order -- a key (rank, ordinal) is unique, so the per-row selection
// sort needs no pool order --, the float / double accumulation of g0..g2 row by row, sep_syllables, and the thrown segment
// (stored = -1, still counted).  Rows and syllables land in the epoch's own frame range, as K3b's do; fa_segfix_kernel
// numbers them.  A record whose tables do not fit kFinSmem (or every record with finalize_in_smem = 0) is finalised by warp
// 0 with finalize_segment in HBM.
// =====================================================================================================================
constexpr int kFinThreads = 256;
constexpr int kFinSmem = 64 * 1024;   // 3 CTAs per SM

__global__ void __launch_bounds__(kFinThreads, 3) fa_segfin_kernel(const FaSegmentParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ int s_wi, s_nr, s_nsel, s_thrown, s_wsum[kFinThreads / 32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const unsigned lt = (1u << lane) - 1u;
  const int maxp = p.maxp;
  const int n_work = *reinterpret_cast<volatile int*>(p.work_count);
  for (;;) {
    if (tid == 0) s_wi = atomicAdd(p.work_count + 1, 1);
    __syncthreads();
    const int wi = s_wi;
    __syncthreads();   // every thread has read s_wi before thread 0 takes the next item
    if (wi >= n_work) break;
    const int2 wk = p.work[wi];
    const int u = wk.x;
    if (p.overflow[u]) continue;        // handed to the general kernel (2) or failed (1): nothing of it is kept
    const FaEpoch E = p.epochs[p.frame_off[u] + u + wk.y];
    Bases bs;
    bs.row0 = p.frame_off[u];
    bs.F = (int)(p.frame_off[u + 1] - bs.row0);
    bs.sb = bs.row0 + u;
    bs.tb = p.track_base[u] + E.trk_off;
    bs.tcap = E.trk_cap;
    bs.pb = (bs.row0 + E.first) * maxp;
    bs.rb = bs.sb + E.first;
    bs.u = u;
    bs.spill = 0;
    const int T = E.n_tr, NP = E.n_pts, len = E.n_arg - E.no_fm_segs;
    auto in_hbm = [&]() {
      if (warp == 0) {
        ScanState st;
        st.current_frame = E.current_frame; st.no_fm_segs = E.no_fm_segs; st.c_ci = E.c_ci; st.c_started = 2; st.w = 0; st.k = 0;
        st.y = E.y; st.v = E.v; st.x = E.y; st.v0 = E.v; st.T = 0; st.s_energy = E.s_energy; st.c_energy = E.c_energy;
        st.n_tr = T; st.n_pts = NP; st.n_slots = 0;
        st.n_segs = wk.y; st.n_stored = 0; st.n_rows = E.first; st.n_syls = E.first; st.overflow = 0;
        finalize_segment(p, st, bs, E.n_arg, lane);
      }
    };
    // layout: rc, ro, fill i32[len] | rank i16[T] | slot i8[T] | cmean f64[nr] | cidx i32[nr] | order i16[nr] |
    //         key u64[n_sel] | e f64[n_sel] | binspan i32[n_sel]     (nr: eligible tracks, n_sel: selected points)
    const int off_tr = 12 * len, off_c = (off_tr + 3 * T + 7) & ~7;
    if (!p.finalize_in_smem || off_c > kFinSmem) { in_hbm(); continue; }
    int* rc = reinterpret_cast<int*>(smem_raw);
    int* ro = rc + len;
    int* fill = ro + len;
    short* rank = reinterpret_cast<short*>(smem_raw + off_tr);
    signed char* slot = reinterpret_cast<signed char*>(rank + T);
    const double vmin = E.v;
    // ---- get_ranked_formants @B35670: count >= 2, mean >= 7, stable ascending by mean ----
    for (int i = tid; i < T; i += kFinThreads) {
      const double m = p.trk_sum_eb[bs.tb + i] / p.trk_sum_e[bs.tb + i];
      slot[i] = p.trk_count[bs.tb + i] >= 2 && m >= 7 ? 1 : -1;    // eligible (slot assigned below)
    }
    for (int r = tid; r < len; r += kFinThreads) { rc[r] = 0; fill[r] = 0; }
    if (tid == 0) { s_nr = 0; s_nsel = 0; s_thrown = 0; }
    __syncthreads();
    {
      int cnt = 0;
      for (int i = tid; i < T; i += kFinThreads) cnt += slot[i] > 0;
      cnt = __reduce_add_sync(FULL, cnt);
      if (lane == 0 && cnt) atomicAdd(&s_nr, cnt);
    }
    __syncthreads();
    const int nr = s_nr;
    const int off_i = off_c + 8 * nr, off_o = off_i + 4 * nr, off_k = (off_o + 2 * nr + 7) & ~7;
    if (off_k > kFinSmem) { in_hbm(); continue; }
    double* cmean = reinterpret_cast<double*>(smem_raw + off_c);
    int* cidx = reinterpret_cast<int*>(smem_raw + off_i);
    short* order = reinterpret_cast<short*>(smem_raw + off_o);
    // the eligible tracks compacted in creation order (block-wide scan of the flags, 256 tracks at a time)
    for (int i0 = 0, base = 0; i0 < T; i0 += kFinThreads) {
      const int i = i0 + tid;
      const bool elig = i < T && slot[i] > 0;
      const unsigned em = __ballot_sync(FULL, elig);
      if (lane == 0) s_wsum[warp] = __popc(em);
      __syncthreads();
      int pre = base, tot = 0;
      for (int w = 0; w < kFinThreads / 32; w++) { if (w < warp) pre += s_wsum[w]; tot += s_wsum[w]; }
      if (elig) {
        const int k = pre + __popc(em & lt);
        cmean[k] = p.trk_sum_eb[bs.tb + i] / p.trk_sum_e[bs.tb + i];
        cidx[k] = i;
        slot[i] = -1;
      }
      base += tot;
      __syncthreads();
    }
    for (int k = tid; k < nr; k += kFinThreads) {
      const double m = cmean[k];
      int rk = 0;
      for (int j = 0; j < nr; j++) {
        const double mj = cmean[j];
        rk += (mj < m || (mj == m && j < k)) ? 1 : 0;   // the compacted list keeps the tracks in creation order
      }
      rank[cidx[k]] = (short)rk;
      order[rk] = (short)k;
    }
    __syncthreads();
    // ---- slot assignment of straighten_formants @B35074 (sequential over the ranking) ----
    if (tid == 0) {
      double anchor = 0;
      int sl = 0;
      for (int r = 0; r < nr; r++) {
        const int k = order[r];
        const double m = cmean[k];
        if (fabs(m - anchor) > 20) {
          anchor = m;
          sl++;
          if (sl >= 3) break;
        }
        slot[cidx[k]] = (signed char)sl;
      }
    }
    __syncthreads();
    // ---- rows: count the selected points of every row; a selected point outside the segment throws ----
    {
      bool thrown = false;
      int nsel = 0;
      for (int q = tid; q < NP; q += kFinThreads) {
        const int i = __ldg(p.pt_track + bs.pb + q), fr = __ldg(p.pt_frame + bs.pb + q);
        if (slot[i] >= 0) {
          if (fr < 0 || fr >= len) thrown = true;   // r[d] is undefined -> TypeError -> .catch(L(-1))
          else { atomicAdd(&rc[fr], 1); nsel++; }
        }
      }
      if (thrown) s_thrown = 1;
      nsel = __reduce_add_sync(FULL, nsel);
      if (lane == 0 && nsel) atomicAdd(&s_nsel, nsel);
    }
    __syncthreads();
    fa_segment seg;
    seg.start = E.current_frame - len; seg.len = len; seg.stored = -1; seg.n_syllables = 0; seg.first_syllable = -1;
    seg.row_offset = -1; seg.ymax = E.y; seg.vmin = E.v; seg.cs_ratio = E.c_energy / E.s_energy;
    if (s_thrown) {
      if (tid == 0) p.segs[bs.sb + wk.y] = seg;
      continue;
    }
    const int n_sel = s_nsel;
    if (off_k + 20 * n_sel > kFinSmem) { in_hbm(); continue; }
    unsigned long long* key = reinterpret_cast<unsigned long long*>(smem_raw + off_k);
    double* pe = reinterpret_cast<double*>(key + n_sel);
    int* bsp = reinterpret_cast<int*>(pe + n_sel);
    if (warp == 0) {   // exclusive prefix of the row counts
      int run = 0;
      for (int r0 = 0; r0 < len; r0 += 32) {
        const int r = r0 + lane;
        const int c = r < len ? rc[r] : 0;
        int incl = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const int t = __shfl_up_sync(FULL, incl, o);
          if (lane >= o) incl += t;
        }
        if (r < len) ro[r] = run + incl - c;
        run += __shfl_sync(FULL, incl, 31);
      }
    }
    __syncthreads();
    // key = rank << 42 | ordinal << 22 | staged index << 2 | slot  (ordinal < 2^20 points, staged index < 2^20, slot < 3)
    for (int q = tid; q < NP; q += kFinThreads) {
      const int i = __ldg(p.pt_track + bs.pb + q);
      const int sl = slot[i];
      if (sl >= 0) {
        const int fr = __ldg(p.pt_frame + bs.pb + q), od = __ldg(p.pt_ord + bs.pb + q);
        const int pos = ro[fr] + atomicAdd(&fill[fr], 1);
        key[pos] = ((unsigned long long)rank[i] << 42) | ((unsigned long long)od << 22) | ((unsigned long long)pos << 2) |
                   (unsigned long long)sl;
        pe[pos] = __ldg(p.pt_e + bs.pb + q);
        bsp[pos] = __ldg(p.pt_binspan + bs.pb + q);
      }
    }
    __syncthreads();
    // ---- apply: thread per row, points in (track rank, point ordinal) order ----
    float* Fout = p.formants + (size_t)(bs.row0 + E.first) * 9;
    float* Eout = p.energy + (size_t)(bs.row0 + E.first) * 3;
    for (int fr = tid; fr < len; fr += kFinThreads) {
      const int k = rc[fr], off = ro[fr];
      float f0 = 0, f1 = 0, f2 = 0, f3 = 0, f4 = 0, f5 = 0, f6 = 0, f7 = 0, f8 = 0, g0 = 0, g1 = 0, g2 = 0;
      long long last = -1;
      for (int it = 0; it < k; it++) {
        long long bestkey = 0x7fffffffffffffffll;
        for (int z = 0; z < k; z++) {
          const long long kz = (long long)key[off + z];
          if (kz > last && kz < bestkey) bestkey = kz;
        }
        last = bestkey;
        const int bq = (int)((bestkey >> 2) & 0xfffffu);
        int sl = (int)(bestkey & 3u);
        const int bs_ = bsp[bq];
        const int bin = bs_ & 0xff, span = bs_ >> 16;   // bits 8..15: the point's lower bound (level 3)
        const double Ep = pe[bq];
        const float cur = sl == 0 ? f0 : sl == 1 ? f3 : f6;
        if ((double)cur > vmin && (double)cur < (double)bin && sl < 2) sl++;
        const float fb = (float)bin, fe = (float)Ep, fs = (float)span;
        if (sl == 0) { f0 = fb; f1 = fe; f2 = fs; }
        else if (sl == 1) { f3 = fb; f4 = fe; f5 = fs; }
        else { f6 = fb; f7 = fe; f8 = fs; }
        g0 = (float)((double)g0 + (double)bin * Ep);
        g1 = (float)((double)g1 + Ep);
        g2 = (float)((double)g2 + (double)span * Ep);
      }
      float* fo = Fout + (size_t)fr * 9;
      fo[0] = f0; fo[1] = f1; fo[2] = f2; fo[3] = f3; fo[4] = f4; fo[5] = f5; fo[6] = f6; fo[7] = f7; fo[8] = f8;
      float* eo = Eout + (size_t)fr * 3;
      eo[0] = g0; eo[1] = g1; eo[2] = g2;
      fill[fr] = (double)g1 > vmin ? 1 : 0;   // sep_syllables needs "energy > vmin" per row
    }
    __syncthreads();
    if (warp != 0) continue;
    // ---- sep_syllables @B34757 (provisional: stored_seg 0, syllables from the epoch's first frame on) ----
    int nsyl = 0;
    if (p.level == 10 || p.level == 11 || p.level == 12 || p.level == 13) {
      int sstart = -1, quiet = 0, loud = 0;
      for (int e0 = 0; e0 < len; e0 += 32) {
        const int e = e0 + lane;
        const bool is_loud = e < len && fill[e] != 0;
        const unsigned bits = __ballot_sync(FULL, is_loud);
        const int cnt = min(32, len - e0);
        for (int b = 0; b < cnt; b++) {
          const int ee = e0 + b;
          if ((bits >> b) & 1u) { quiet = 0; loud++; if (sstart < 0) sstart = ee; }
          else quiet++;
          if ((loud > 20 && quiet > 0) || (loud > 10 && quiet > 1) || (loud > 0 && quiet > 4) || (ee >= len - 1 && loud > 4)) {
            const int end = ee - quiet;
            if (end - sstart > 1) {
              if (lane == 0) {
                fa_syllable sy;
                sy.stored_seg = 0; sy.start = sstart; sy.len = end - sstart; sy.reserved = 0;
                p.syls[bs.sb + E.first + nsyl] = sy;
              }
              nsyl++;
              sstart = -1;
              loud = 0;
            }
          }
        }
      }
    }
    if (lane == 0) {
      seg.stored = 0; seg.row_offset = E.first; seg.first_syllable = E.first; seg.n_syllables = nsyl;
      p.segs[bs.sb + wk.y] = seg;
    }
  }
}

__global__ void __launch_bounds__(kCtlWarps * 32) fa_segfix_kernel(const FaSegmentParams p) {
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int ui = blockIdx.x * kCtlWarps + wib;
  if (ui >= p.utt_count) return;
  const int u = p.utt_begin + ui;
  const long long row0 = p.frame_off[u], sb = row0 + u;
  const int nseg = p.n_segs[u];
  int k = 0, rows = 0, nsyl = 0;
  if (!p.overflow[u]) {
    for (int si = 0; si < nseg; si++) {
      fa_segment sg = p.segs[sb + si];
      if (sg.stored < 0) continue;       // dropped by the throw: seg_ci keeps it, nothing was stored
      // the formant / energy rows stay where K3b put them (the epoch's first frame): K4 / K6 / K5 find them through the
      // epoch table, and the dense gather (K5) copies them segment by segment with many CTAs -- moving 136 k rows of a
      // one-hour stream down in place with one warp took 23 ms
      const int ssrc = sg.first_syllable;
      for (int j0 = 0; j0 < sg.n_syllables; j0 += 32) {
        const int j = j0 + lane;
        fa_syllable sy;
        if (j < sg.n_syllables) { sy = p.syls[sb + ssrc + j]; sy.stored_seg = k; }
        __syncwarp();
        if (j < sg.n_syllables) p.syls[sb + nsyl + j] = sy;
        __syncwarp();
      }
      if (lane == 0) {
        sg.stored = k; sg.row_offset = rows; sg.first_syllable = nsyl;
        p.segs[sb + si] = sg;
      }
      k++; rows += sg.len; nsyl += sg.n_syllables;
    }
  }
  if (lane == 0) { p.n_stored[u] = k; p.n_rows[u] = rows; p.n_syls[u] = nsyl; }
}

}  // namespace

cudaError_t fa_launch_segment(const FaSegmentParams& p_in, cudaStream_t s, int* launches) {
  if (p_in.utt_count <= 0) return cudaSuccess;
  FaSegmentParams p = p_in;
  const int kw = p.warps_per_cta >= 1 && p.warps_per_cta <= 4 ? p.warps_per_cta : kWarps;
  // per-warp shared-memory slice = the struct.  (Extra scratch behind it for finalize_fast was tried: 56 KB per CTA x 4 CTAs
  // per SM leaves ~4 KB of L1 for the candidate / pool reads and the stack, and every variant of the scan lost 0.35 ms.)
  p.smem_per_warp = (int)sizeof(WarpShared);
  const int bytes = p.smem_per_warp * kw;
  const int regs = p.reg_cap > 0 ? p.reg_cap : 255;
  if (p.mode == 1) {
    if (p.ctl_chunk > 0) {
      if (p.n_cchunks > 0) fa_segctl_chunk_kernel<<<(p.n_cchunks + kCtlWarps - 1) / kCtlWarps, kCtlWarps * 32, 0, s>>>(p);
      fa_segctl_verify_kernel<<<(p.utt_count + kCtlWarps - 1) / kCtlWarps, kCtlWarps * 32, 0, s>>>(p);
      if (launches) (*launches)++;
    } else {
      fa_segctl_kernel<<<(p.utt_count + kCtlWarps - 1) / kCtlWarps, kCtlWarps * 32, 0, s>>>(p);
    }
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    const int grid = (p.n_workers + kw - 1) / kw;
    auto launch = [&](auto kernel) -> cudaError_t {
      cudaError_t e2 = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
      if (e2 != cudaSuccess) return e2;
      kernel<<<grid, kw * 32, bytes, s>>>(p);
      return cudaGetLastError();
    };
    e = regs <= 64 ? launch(fa_segtrack_kernel<1024>) : regs <= 96 ? launch(fa_segtrack_kernel<640>) : launch(fa_segtrack_kernel<128>);
    if (e != cudaSuccess) return e;
    fa_segfix_kernel<<<(p.utt_count + kCtlWarps - 1) / kCtlWarps, kCtlWarps * 32, 0, s>>>(p);
    if (launches) (*launches) += 3;
    return cudaGetLastError();
  }
  const int grid = (p.utt_count + kw - 1) / kw;
  auto launch = [&](auto kernel) -> cudaError_t {
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e != cudaSuccess) return e;
    kernel<<<grid, kw * 32, bytes, s>>>(p);
    return cudaGetLastError();
  };
  cudaError_t e = cudaSuccess;
  if (p.impl == 3) {   // the two-warp pipeline; whatever it hands back (overflow == 2) is redone by the general kernel below
    p.redo_only = 0;
    const int pbytes = kPipeUtts * (p.smem_per_warp + (int)sizeof(PipeShared));
    e = cudaFuncSetAttribute(fa_segment3_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, pbytes);
    if (e != cudaSuccess) return e;
    fa_segment3_kernel<<<(p.utt_count + kPipeUtts - 1) / kPipeUtts, 2 * kPipeUtts * 32, pbytes, s>>>(p);
    e = cudaGetLastError();
    if (launches) (*launches)++;
    if (e != cudaSuccess) return e;
    p.redo_only = 1;
  } else if (p.impl == 2) {
    p.redo_only = 0;
    // The fast kernel never touches the general kernel's score table at the end of WarpShared: its slice is kSlimBytes, so that
    // 16 warps fit an SM's shared memory.  Registers: 153 by default; a launch with more warps than one resident wave of those
    // (12 per SM) is throughput bound -- the 128-register build (launch bound 480: no spills, 1 % slower alone) keeps 16 warps
    // per SM resident instead of 12.  FA_K3_REGS forces a cap through the launch bound (65536 / bound, rounded down to a
    // multiple of 8): 64, 96, 128 (<= 144), else the default.
    static int num_sms = 0;
    if (!num_sms) {
      int dev = 0;
      cudaGetDevice(&dev);
      cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev);
    }
    const int regs2 = p.reg_cap > 0 ? p.reg_cap : (p.utt_count > num_sms * 12 ? 128 : 255);
    const int full = p.smem_per_warp;
    p.smem_per_warp = kSlimBytes;
    auto launch2 = [&](auto kernel) -> cudaError_t {
      cudaError_t e2 = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSlimBytes * kw);
      if (e2 != cudaSuccess) return e2;
      kernel<<<grid, kw * 32, kSlimBytes * kw, s>>>(p);
      return cudaGetLastError();
    };
    e = regs2 <= 64 ? launch2(fa_segment2_kernel<1024>) : regs2 <= 96 ? launch2(fa_segment2_kernel<640>)
        : regs2 <= 144 ? launch2(fa_segment2_kernel<480>) : launch2(fa_segment2_kernel<128>);
    p.smem_per_warp = full;
    if (launches) (*launches)++;
    if (e != cudaSuccess) return e;
    if (p.level != 3) {   // the recorded finalisations, then the numbering of the stores (level 3 finalised in the chain)
      e = cudaFuncSetAttribute(fa_segfin_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kFinSmem);
      if (e != cudaSuccess) return e;
      fa_segfin_kernel<<<num_sms * 3, kFinThreads, kFinSmem, s>>>(p);
      fa_segfix_kernel<<<(p.utt_count + kCtlWarps - 1) / kCtlWarps, kCtlWarps * 32, 0, s>>>(p);
      if (launches) (*launches) += 2;
      e = cudaGetLastError();
      if (e != cudaSuccess) return e;
    }
    p.redo_only = 1;   // whatever fa_segment2_kernel handed back (overflow == 2): normally nothing, every warp exits at once
  } else {
    p.redo_only = 0;
  }
  e = regs <= 64 ? launch(fa_segment_kernel<1024>) : regs <= 96 ? launch(fa_segment_kernel<640>) : launch(fa_segment_kernel<128>);
  if (launches) (*launches)++;
  return e;
}
