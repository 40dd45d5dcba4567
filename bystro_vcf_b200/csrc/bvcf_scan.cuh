// bvcf_scan.cuh -- north-star kernels (1)+(3) fused: newline/tab index + per-sample genotype classify.
//
// One warp streams one byte range of the input exactly once (cp.async 16-byte loads into a per-warp
// shared-memory ring, 512 B per step), finds line boundaries and tab counts with SWAR byte compares +
// __ballot_sync/__popc + warp prefix sums, and classifies every sample's GT token on the fly.  It owns the
// lines that START in its range (it reads past the range end to finish the last one).  Products:
//   * LineRec per record with the header's field count (main.go:449 len(record)==len(header)), including the
//     offsets of its first nine tabs (the field index the rows kernel needs) and the ALT #1 genotype
//     summary (het/hom/missing counts, ac, an -- main.go:1042-1194),
//   * one 32-bit event per non-reference sample, in header order (main.go:1057 loop order), from which the
//     names kernel writes the het/hom/missing lists (and the stats kernel serves the other ALT numbers).
// Replaces: strings.Split (main.go:535) + the sample loop of makeHetHomozygotes (main.go:1057-1191).
//
// Three tiers per 512-byte window, chosen warp-uniformly:
//   T1  all 128 fields are "0|0\t" (or "0/0\t")  -> 5 XOR/OR on the raw words + vote, nothing else
//   T2  all 128 fields are "x|y\t" with x,y in [0-9.] -> SWAR classify in registers, ordered compaction of events
//   T3  anything else (line start/end, fixed fields, FORMAT suffixes, odd widths): tab/newline masks, ballots
//       and prefix sums; its sample zone is still classified with the T2 vector code when it is regular,
//       field by field otherwise
#pragma once
#include "bvcf_common.cuh"

namespace bvcf {

constexpr int WIN = 512;                 // bytes per warp step
constexpr int STAGES = 8;                // ring stages per warp
constexpr int RING = WIN * STAGES;       // 4 KiB per warp
constexpr int PF_PAIRS = 3;              // pairs of windows in flight beyond the pair being read
constexpr int SCAN_WARPS = 8;            // warps per CTA
constexpr int FS_NONE = 0x7FFFFFFF;      // "inside a field": no known field start

struct ScanParams {
  const uint8_t *in;        // region base (>= 16-byte aligned)
  uint64_t begin, end;      // data lines live in [begin, end); in[end-1] == '\n'
  uint64_t buf_len;         // readable bytes from `in`: multiple of 512 and >= round_up(end,512)+512
  uint64_t a0;              // begin & ~511: ranges tile [a0, ...)
  uint32_t range_bytes;     // multiple of 512
  uint32_t r0, n_ranges;    // this launch handles global ranges [r0, r0+n_ranges)
  uint32_t slots_per_range, evcap_words;
  LineRec *recs;            // n_ranges * slots_per_range
  uint32_t *range_nrec;     // records per range
  uint32_t *range_nlines;   // all newline-terminated lines that start in the range
  uint32_t *events;         // n_ranges * evcap_words
  RunCounters *ctr;
  int H, eol_width;
};

// per-line accumulators; *_l are per-lane partial sums reduced when the line ends
struct LineAcc {
  uint32_t an_l, an_uni;    // non-missing allele count (main.go:1067,1169)
  uint32_t het_l, hom_l;    // ALT #1 heterozygotes / homozygotes (main.go:1080-1109,1185)
  uint32_t ac_l;            // ALT #1 allele count
  uint32_t miss_l;          // missing samples (main.go:1113,1150)
  uint32_t flag_l;          // 1: an event carries another ALT number or needs the general GT grammar
};

struct WarpState {
  uint64_t line_start;
  int fsr;                  // first unprocessed field start, relative to the current window; FS_NONE inside a field
  uint32_t col;             // field index of the field at fsr == tabs of this line before it
  uint32_t ev_w, line_ev_start;  // event write cursor (words, relative to this range's slice)
  uint32_t nrec, nlines;
  uint32_t refpat;          // "0|0\t" or "0/0\t", follows the data's separator
  int mode;                 // 0 seeking the first line start, 1 inside an owned line, 2 done
  LineAcc a;
};

__device__ __forceinline__ uint4 lds128(uint32_t a) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];\n" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
  return v;
}
__device__ __forceinline__ uint32_t lds32(uint32_t a) {
  uint32_t v;
  asm volatile("ld.shared.u32 %0, [%1];\n" : "=r"(v) : "r"(a));
  return v;
}

__device__ __forceinline__ uint32_t bits_range16(int lo, int hi) {  // bits [lo, hi) clipped to [0,16)
  lo = lo < 0 ? 0 : lo;
  hi = hi > 16 ? 16 : hi;
  return hi <= lo ? 0u : (((1u << hi) - 1u) & ~((1u << lo) - 1u));
}

__device__ __forceinline__ uint32_t tok_code(uint32_t c) {  // single-character allele token
  uint32_t d = c - '0';
  return c == '.' ? EV_CODE_MISSING : (d <= 9 ? d : 0u);
}

__device__ __forceinline__ void start_line(WarpState &st, uint64_t start, int rel) {
  st.line_start = start; st.fsr = rel; st.col = 0;
  st.a.an_l = st.a.an_uni = st.a.het_l = st.a.hom_l = st.a.ac_l = st.a.miss_l = st.a.flag_l = 0;
  st.line_ev_start = st.ev_w;
}

// ALT #1 bookkeeping for one fast-classified sample with allele codes c1,c2 (c2 == EV_CODE_ABSENT: haploid)
__device__ __forceinline__ void acc_sample(LineAcc &a, uint32_t c1, uint32_t c2) {
  const uint32_t hap = c2 == EV_CODE_ABSENT;
  const uint32_t alt = (c1 == 1) + (c2 == 1);
  a.ac_l += alt;
  a.hom_l += hap ? alt : (alt >> 1);
  a.het_l += hap ? 0u : (alt & 1u);
  a.flag_l |= (c1 > 1) | (!hap && c2 > 1);
}

// ---- the T2 vector code: four realigned fields per lane, XORed with the reference pattern -------------
// t[j] == 0: reference genotype.  Structure (separator, tab) already verified by the caller; allele bytes are
// digits (t byte <= 9) or, when `dots`, '.' (0x1E).  Words outside the sample zone arrive zeroed.
// The lane's four fields become ONE quad event (eight 4-bit allele codes, bvcf_common.cuh): no per-sample
// loop, the compaction is a ballot + popc, the ALT #1 summary is nibble-parallel arithmetic.
__device__ __forceinline__ uint32_t pack_quad(const uint32_t t[4], bool dots) {
  if (dots) {
    const uint32_t K = 0x000F000Fu;  // '.' ^ '0' = 0x1E -> nibble 0xE
    return (t[0] & K) | ((t[1] & K) << 4) | ((t[2] & K) << 8) | ((t[3] & K) << 12);
  }
  return t[0] | (t[1] << 4) | (t[2] << 8) | (t[3] << 12);  // digits: every allele byte is already a nibble
}
__device__ __forceinline__ uint32_t nibbles_eq(uint32_t pl, uint32_t rep) {  // bit 3 of every nibble equal to rep's
  const uint32_t y = pl ^ rep;
  return ~(((y & 0x77777777u) + 0x77777777u) | y) & 0x88888888u;
}
// ALT #1 bookkeeping of the quad payloads of two windows (diploid fields only: the vector path; pb = 0 for one
// window).  Window B's marks are moved one bit below A's, so one popc counts both.
__device__ __forceinline__ void acc_quad_pair(LineAcc &a, uint32_t pa, uint32_t pb, bool dots) {
  uint32_t oa = nibbles_eq(pa, 0x11111111u), ob = nibbles_eq(pb, 0x11111111u);
  if (dots) {
    const uint32_t da = nibbles_eq(pa, 0xEEEEEEEEu), db = nibbles_eq(pb, 0xEEEEEEEEu);
    const uint32_t fa = (da | (da >> 16)) & 0x8888u, fb = (db | (db >> 16)) & 0x8888u;  // samples with a '.' token:
    const uint32_t nm = __popc(fa | (fb >> 1));                                        // missing (main.go:1113,1150)
    a.miss_l += nm;
    a.an_l -= 2 * nm;
    const uint32_t ga = ((fa | (fa << 16)) >> 3) * 15u, gb = ((fb | (fb << 16)) >> 3) * 15u;  // both nibbles of them
    oa &= ~ga; ob &= ~gb;
    pa &= ~ga; pb &= ~gb;
  }
  const uint32_t one = oa | (ob >> 1);
  const uint32_t n1 = __popc(one), n2 = __popc(one & (one >> 16));
  a.ac_l += n1;
  a.hom_l += n2;
  a.het_l += n1 - 2 * n2;
  a.flag_l |= (pa | pb) & 0xEEEEEEEEu;  // nibbles >= 2
}
__device__ __forceinline__ void classify_push_words4(const ScanParams &p, WarpState &st, uint32_t *my_events,
                                                     const uint32_t t[4], int samp0, bool dots, int lane) {
  const uint32_t pl = pack_quad(t, dots);
  const uint32_t bal = __ballot_sync(FULL, pl != 0);
  if (bal == 0) return;
  const uint32_t n = 2 * __popc(bal);
  if (st.ev_w + n <= p.evcap_words) {
    if (pl)
      *reinterpret_cast<uint2 *>(my_events + st.ev_w + 2 * __popc(bal & ((1u << lane) - 1u))) =
          make_uint2((uint32_t)(samp0 + (int)EV_BASE_BIAS), pl);
  } else if (lane == 0) {
    p.ctr->ev_overflow = 1;
  }
  acc_quad_pair(st.a, pl, 0u, dots);
  st.ev_w += n;
}

// Two adjacent windows at once: the quads of window A (all lanes) precede those of window B.
__device__ __forceinline__ void classify_push_pair(const ScanParams &p, WarpState &st, uint32_t *my_events,
                                                   const uint32_t ta[4], const uint32_t tb[4], int samp0, bool dots,
                                                   int lane) {
  const uint32_t pa = pack_quad(ta, dots), pb = pack_quad(tb, dots);
  const uint32_t ba = __ballot_sync(FULL, pa != 0), bb = __ballot_sync(FULL, pb != 0);
  if ((ba | bb) == 0) return;
  const uint32_t qa = __popc(ba), n = 2 * (qa + __popc(bb));
  if (st.ev_w + n <= p.evcap_words) {
    uint2 *dst = reinterpret_cast<uint2 *>(my_events + st.ev_w);  // one address for both stores
    const uint32_t lt = (1u << lane) - 1u, e = (uint32_t)(samp0 + (int)EV_BASE_BIAS);
    if (pa) dst[__popc(ba & lt)] = make_uint2(e, pa);
    if (pb) dst[qa + __popc(bb & lt)] = make_uint2(e + 128u, pb);
  } else if (lane == 0) {
    p.ctr->ev_overflow = 1;
  }
  acc_quad_pair(st.a, pa, pb, dots);
  st.ev_w += n;
}

// SWAR validity of four XORed fields: separator/tab bytes unchanged, allele bytes digits (or '.')
// Quick test on the OR of the words (no false negatives: the OR of nibbles is >= each of them; a false positive,
// e.g. alleles 8 and 2 in one lane, only costs the exact test below).
__device__ __forceinline__ uint32_t bad_digits4(const uint32_t t[4], uint32_t keep_mask3) {
  const uint32_t o = t[0] | t[1] | t[2] | (t[3] & keep_mask3);
  return (o & 0xFFF0FFF0u) | (((o & 0x000F000Fu) + 0x00060006u) & 0x00100010u);
}
__device__ __forceinline__ uint32_t bad_digits8(const uint32_t ta[4], const uint32_t tb[4]) {
  const uint32_t o = ta[0] | ta[1] | ta[2] | ta[3] | tb[0] | tb[1] | tb[2] | tb[3];
  return (o & 0xFFF0FFF0u) | (((o & 0x000F000Fu) + 0x00060006u) & 0x00100010u);
}
// Exact test with '.' allowed: every allele byte (XORed with '0') is 0..9 or 0x1E, every other byte 0.
// With all bytes below 0x20 (first term), b + 22 carries into bit 5 iff b >= 10, b + 2 iff b >= 30, b + 1 iff b == 31:
// bad iff 10 <= b <= 29 or b == 31.
__device__ __forceinline__ uint32_t bad_digits_or_dots4(const uint32_t t[4], uint32_t keep_mask3) {
  const uint32_t o = t[0] | t[1] | t[2] | (t[3] & keep_mask3);
  uint32_t acc = 0;
#pragma unroll
  for (int j = 0; j < 4; j++) {
    const uint32_t x = t[j] + 0x00160016u, y = t[j] + 0x00020002u, z = t[j] + 0x00010001u;
    acc |= (x & ~y) | z;
  }
  return (o & 0xFFE0FFE0u) | (acc & 0x00200020u);
}

// ---- T3: the general window ------------------------------------------------------------------------
template <bool HAS_SAMPLES>
__device__ __forceinline__ void scan_window_general(const ScanParams &p, WarpState &st, uint32_t ring_base_s,
                                                    uint32_t stage_off, const uint4 &v, uint64_t pos, uint64_t rend,
                                                    int lane, LineRec *my_recs, uint32_t *my_events) {
  const bool eol2 = p.eol_width == 2;
  const uint32_t tm = eq_mask16(v, 0x09090909u);
  uint32_t nm = eq_mask16(v, 0x0A0A0A0Au);  // newlines not yet consumed: each segment takes the lowest one

  int seg_lo = 0;
  if (st.mode == 1 && st.fsr != FS_NONE && st.fsr > 0) {  // bytes before the field start are consumed
    seg_lo = st.fsr;
    nm &= bits_range16(seg_lo - lane * 16, 16);
  }

  while (seg_lo < WIN) {
    // first newline at or after seg_lo
    const int lo_l = seg_lo - lane * 16;
    const uint32_t ball = __ballot_sync(FULL, nm != 0);
    int nl = WIN;
    if (ball) {
      const int l = __ffs(ball) - 1;
      const uint32_t m = __shfl_sync(FULL, nm, l);
      nl = l * 16 + __ffs(m) - 1;
      if (lane == l) nm &= nm - 1;
    }
    if (st.mode == 0) {  // seeking the first owned line start
      if (nl == WIN) return;
      const uint64_t start = pos + nl + 1;
      if (start >= rend) { st.mode = 2; return; }
      st.mode = 1;
      start_line(st, start, nl + 1);
      seg_lo = nl + 1;
      continue;
    }
    // tabs of this segment: bytes [seg_lo, nl)
    int tab_hi = nl;
    if (eol2 && nl < WIN && nl > 0) tab_hi = nl - 1;  // row[:len-2] strips the byte before '\n' (main.go:535)
    const uint32_t tm_l = tm & bits_range16(lo_l, tab_hi - lane * 16);
    const uint32_t cnt = __popc(tm_l);
    // the per-lane field index (prefix sum) is only needed while the fixed fields go by, or field by field
    // below; a segment that lies in the sample zone just needs its tab count (one REDUX)
    uint32_t excl = 0, total;
    bool have_excl = false;
    if (st.col < 9) {
      const uint32_t incl = warp_incl_scan(cnt, lane);
      excl = incl - cnt;
      total = __shfl_sync(FULL, incl, 31);
      have_excl = true;
    } else {
      total = __reduce_add_sync(FULL, cnt);
    }

    // field index: offsets of the record's first nine tabs (strings.Split, main.go:535)
    if (st.col < 9 && st.nrec < p.slots_per_range) {
      uint16_t *const tabp = my_recs[st.nrec].tab;
      const uint32_t off0 = (uint32_t)(pos - st.line_start) + (uint32_t)(lane * 16);  // a line is < 4 GiB (LineRec.len)
      uint32_t m = tm_l;
      uint32_t idx = st.col + excl;
      while (m && idx < 9) {
        const uint32_t off = off0 + (uint32_t)(__ffs(m) - 1);
        m &= m - 1;
        tabp[idx] = off < 0xFFFFu ? (uint16_t)off : (uint16_t)0xFFFFu;
        idx++;
      }
    }

    int nfs = FS_NONE;       // hand-over to the next window when this segment reaches the window end
    uint32_t col_extra = 0;
    if (HAS_SAMPLES) {
      // ---- where do this segment's sample fields begin? ----
      int s9 = -1;           // window-relative start of the first sample field of the segment
      uint32_t samp_base = 0;
      if (st.col >= 9) {
        if (st.fsr == seg_lo) { s9 = seg_lo; samp_base = st.col - 9; }
      } else if (st.col + total >= 9) {
        const uint32_t k9 = 8 - st.col;  // in-segment index of the ninth tab
        const bool mine = k9 >= excl && k9 < excl + cnt;
        const uint32_t who = __ballot_sync(FULL, mine);
        int pos9 = 0;
        if (mine) {  // the (k9 - excl)-th set bit of tm_l: drop the lower ones
          uint32_t m9 = tm_l;
          for (uint32_t d = k9 - excl; d > 0; d--) m9 &= m9 - 1;
          pos9 = lane * 16 + __ffs(m9) - 1;
        }
        s9 = __shfl_sync(FULL, pos9, __ffs(who) - 1) + 1;
      }
      const int zone_end = nl;  // sample fields of this segment live in [s9, zone_end)
      bool vector_ok = false;
      if (s9 >= 0 && s9 < zone_end && !(eol2 && nl < WIN)) {
        // ---- regular zone? classify it with the T2 vector code ----
        const uint32_t w4 = lds32(ring_base_s + ((stage_off + lane * 16 + 16) & (RING - 1)));
        const uint32_t sh = (uint32_t)(s9 & 3) * 8u;
        const uint32_t rp = st.refpat;
        uint32_t t[4] = {__funnelshift_r(v.x, v.y, sh) ^ rp, __funnelshift_r(v.y, v.z, sh) ^ rp,
                         __funnelshift_r(v.z, v.w, sh) ^ rp, __funnelshift_r(v.w, w4, sh) ^ rp};
        const int ws0 = lane * 16 + (s9 & 3);  // start of this lane's first realigned word
        // word j of this lane starts at ws0 + 4 j, in phase with s9; it is in the zone iff s9 <= ws < zone_end
        int jlo = (s9 - ws0 + 3) >> 2, jhi = (zone_end - ws0 + 3) >> 2;  // arithmetic shifts: ceilings
        jlo = jlo < 0 ? 0 : jlo;
        jhi = jhi > 4 ? 4 : jhi;
        const uint32_t zone = jhi > jlo ? (((1u << jhi) - 1u) & ~((1u << jlo) - 1u)) : 0u;
#pragma unroll
        for (int j = 0; j < 4; j++) t[j] = (zone >> j) & 1u ? t[j] : 0u;
        bool bad_shape = false;
        if (nl < WIN) {  // the line ends here: where does the newline fall within its field?  (warp-uniform)
          const int r = (nl - s9) & 3;
          if (r == 3) {  // "x|y\n": the last field ends with '\n', not '\t'
            const int jn = (nl - 3 - ws0) >> 2;
#pragma unroll
            for (int j = 0; j < 4; j++) if (j == jn) t[j] ^= 0x03000000u & (0u - ((zone >> j) & 1u));
          } else {
            // r == 1, 2: a short last field; r == 0: an EMPTY last field (a tab right before the newline), one
            // token "" that counts towards an (main.go:1143,1166): both go field by field
            bad_shape = true;
          }
        }
        uint32_t bad = bad_digits4(t, 0xFFFFFFFFu) | (bad_shape ? 1u : 0u);
        bool dots = false;
        if (!__all_sync(FULL, bad == 0)) {
          bad = bad_digits_or_dots4(t, 0xFFFFFFFFu) | (bad_shape ? 1u : 0u);
          dots = true;
        }
        if (__all_sync(FULL, bad == 0)) {
          vector_ok = true;
          const int samp0 = (int)samp_base + ((ws0 - s9) >> 2);  // arithmetic shift: negative before the zone
          st.a.an_l += 2 * __popc(zone);
          classify_push_words4(p, st, my_events, t, samp0, dots, lane);  // out-of-zone words are zero
          if (nl == WIN) {  // zone runs to the window end: the next window continues in the same phase
            const int n_words = (WIN - s9 + 3) >> 2;
            const int ws_last = s9 + 4 * (n_words - 1);
            nfs = ws_last + 4 - WIN;
            col_extra = ws_last + 3 >= WIN ? 1u : 0u;  // that field's tab lies in the next window: pre-count it
          }
        }
      }
      if (!vector_ok) {
        // ---- field by field ----
        if (!have_excl) excl = warp_incl_scan(cnt, lane) - cnt;
        int last_end = -1;   // window-relative index of the '\t' that ends this lane's last field, if known
        uint32_t last_sep = 0;
        const uint32_t prev_hi = __shfl_up_sync(FULL, tm_l >> 15, 1);
        uint32_t fm = ((tm_l << 1) | (lane > 0 ? (prev_hi & 1u) : 0u)) & 0xFFFFu;
        if (st.fsr == seg_lo) {
          const int sl = seg_lo - lane * 16;
          if (sl >= 0 && sl < 16) fm |= 1u << sl;
        }
        const uint32_t fm_all = fm;
        uint32_t evbuf[16];
        int nev = 0;
        while (fm) {
          const int sl = __ffs(fm) - 1;
          fm &= fm - 1;
          const uint32_t fidx = st.col + excl + __popc(tm_l & ((1u << sl) - 1u));
          last_end = -1;
          if (fidx < 9) continue;
          const uint32_t samp = fidx - 9;
          const int s = lane * 16 + sl;
          // 5 bytes at s from the ring (s+4 may reach into the next window: already loaded)
          const uint32_t a = stage_off + (uint32_t)s;
          const uint32_t w0 = lds32(ring_base_s + ((a & ~3u) & (RING - 1)));
          const uint32_t w1 = lds32(ring_base_s + (((a & ~3u) + 4u) & (RING - 1)));
          const uint32_t sh = (a & 3u) * 8u;
          const uint32_t lo = __funnelshift_r(w0, w1, sh);
          const uint32_t b0 = lo & 0xFF, b1 = (lo >> 8) & 0xFF, b2 = (lo >> 16) & 0xFF, b3 = lo >> 24;
          const uint32_t b4 = (w1 >> sh) & 0xFF;
          auto is_end = [&](uint32_t c, uint32_t nx) { return c == '\t' || c == '\n' || c == ':' || (eol2 && nx == '\n'); };
          auto is_sep = [](uint32_t c) { return c == '|' || c == '/'; };
          const bool e0 = is_end(b0, b1), e1 = is_end(b1, b2), e2 = is_end(b2, b3), e3 = is_end(b3, b4);
          if (e0) {  // empty GT: one token "" (main.go:1143,1166)
            st.a.an_l += 1;
            if (b0 == '\t') last_end = s;
          } else if (!is_sep(b0) && e1) {  // haploid, one single-character token
            const uint32_t c = tok_code(b0);
            if (c == EV_CODE_MISSING) {
              evbuf[nev++] = samp + EV_BASE_BIAS; evbuf[nev++] = ev_single_payload(EV_CODE_MISSING, EV_CODE_MISSING);
              st.a.miss_l++;
            } else {
              st.a.an_l += 1;
              if (c) {
                evbuf[nev++] = samp + EV_BASE_BIAS; evbuf[nev++] = ev_single_payload(c, EV_CODE_ABSENT);
                acc_sample(st.a, c, EV_CODE_ABSENT);
              }
            }
            if (b1 == '\t') last_end = s + 1;
          } else if (!is_sep(b0) && is_sep(b1) && !e2 && !is_sep(b2) && e3) {  // diploid x|y or x/y
            const uint32_t c1 = tok_code(b0), c2 = tok_code(b2);
            if (c1 == EV_CODE_MISSING || c2 == EV_CODE_MISSING) {
              evbuf[nev++] = samp + EV_BASE_BIAS; evbuf[nev++] = ev_single_payload(EV_CODE_MISSING, EV_CODE_MISSING);
              st.a.miss_l++;
            } else {
              st.a.an_l += 2;
              if (c1 | c2) {
                evbuf[nev++] = samp + EV_BASE_BIAS; evbuf[nev++] = ev_single_payload(c1, c2);
                acc_sample(st.a, c1, c2);
              }
            }
            if (b3 == '\t') { last_end = s + 3; last_sep = b1; }
          } else {  // general grammar: resolved exactly by the stats/names kernels
            evbuf[nev++] = (samp + EV_BASE_BIAS) | EV_COMPLEX;
            evbuf[nev++] = (uint32_t)(pos + (uint64_t)s - st.line_start);
            st.a.flag_l |= 1;
          }
        }
        // ordered compaction of this segment's events
        const uint32_t eincl = warp_incl_scan((uint32_t)nev, lane);
        const uint32_t etot = __shfl_sync(FULL, eincl, 31);
        if (etot) {
          if (st.ev_w + etot <= p.evcap_words) {
            uint32_t *dst = my_events + st.ev_w + (eincl - nev);
            for (int k = 0; k < nev; k++) dst[k] = evbuf[k];
          } else if (lane == 0) {
            p.ctr->ev_overflow = 1;
          }
          st.ev_w += etot;
        }
        if (nl == WIN) {  // hand the field phase over to the next window
          const uint32_t last_tab = __shfl_sync(FULL, tm_l >> 15, 31) & 1u;
          if (last_tab) {
            nfs = 0;
          } else {
            const uint32_t have = __ballot_sync(FULL, fm_all != 0);
            if (have) {
              const int l = 31 - __clz(have);
              const int le = __shfl_sync(FULL, last_end, l);
              const uint32_t sp = __shfl_sync(FULL, last_sep, l);
              if (le >= WIN) {
                nfs = le + 1 - WIN; col_extra = 1;  // pre-count that tab
                if (sp) st.refpat = 0x09300030u | (sp << 8);
              }
            }
          }
        }
      }
    }
    st.col += total;

    if (nl < WIN) {  // the line ends inside this window
      st.nlines++;
      const LineAcc &a = st.a;
      const uint32_t an = __reduce_add_sync(FULL, a.an_l) + a.an_uni;
      uint32_t n_het = 0, n_hom = 0, n_miss = 0, ac = 0, flag = 0;
      if (HAS_SAMPLES) {
        flag = __any_sync(FULL, a.flag_l != 0);
        if (__any_sync(FULL, (a.het_l | a.hom_l | a.miss_l) != 0)) {
          n_het = __reduce_add_sync(FULL, a.het_l); n_hom = __reduce_add_sync(FULL, a.hom_l);  // REDUX
          ac = __reduce_add_sync(FULL, a.ac_l); n_miss = __reduce_add_sync(FULL, a.miss_l);
        }
      }
      if (st.col == (uint32_t)(p.H - 1)) {
        if (st.nrec < p.slots_per_range) {
          if (lane == 0) {
            LineRec *r = &my_recs[st.nrec];
            r->start = st.line_start;
            r->len = (uint32_t)(pos + nl + 1 - st.line_start);
            r->an = an;
            r->ev_start = st.line_ev_start;
            r->ev_count = st.ev_w - st.line_ev_start;
            r->ord = st.nlines - 1;
            r->flags = (uint16_t)flag;
            r->n_het1 = n_het; r->n_hom1 = n_hom; r->n_miss = n_miss; r->ac1 = ac;
          }
        } else if (lane == 0) {
          p.ctr->slot_overflow = 1;
        }
        st.nrec++;
      } else {
        st.ev_w = st.line_ev_start;  // wrong field count: the line yields nothing (main.go:449)
      }
      const uint64_t start = pos + nl + 1;
      if (start >= rend) { st.mode = 2; return; }
      start_line(st, start, nl + 1);
      seg_lo = nl + 1;
      continue;
    }
    // segment ran to the window end
    st.col += col_extra;
    st.fsr = nfs;
    return;
  }
  // the last segment ended with a newline on the window's final byte: the next line starts the next window
  if (st.mode == 1) st.fsr = seg_lo - WIN;
}

// ---- the kernel ------------------------------------------------------------------------------------
template <bool HAS_SAMPLES>
__global__ void __launch_bounds__(SCAN_WARPS * 32) bvcf_scan_genotype_kernel(const ScanParams p) {
  extern __shared__ __align__(16) uint8_t smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rl = blockIdx.x * SCAN_WARPS + warp;  // range index within this launch
  if (rl >= p.n_ranges) return;
  const uint64_t rstart = p.a0 + (uint64_t)(p.r0 + rl) * p.range_bytes;  // 512-aligned
  uint64_t rend = rstart + p.range_bytes;
  if (rend > p.end) rend = p.end;
  LineRec *my_recs = p.recs + (size_t)rl * p.slots_per_range;
  uint32_t *my_events = p.events + (size_t)rl * p.evcap_words;

  WarpState st;
  st.nrec = 0; st.nlines = 0; st.ev_w = 0;
  st.refpat = 0x09307C30u;  // "0|0\t"
  st.mode = 0;
  start_line(st, 0, FS_NONE);
  if (rstart >= p.end) {
    st.mode = 2;
  } else if (rstart <= p.begin) {  // first range: the region starts with a line
    st.mode = 1; st.line_start = p.begin; st.fsr = (int)(p.begin - rstart);
  } else if (p.in[rstart - 1] == '\n') {
    st.mode = 1; st.line_start = rstart; st.fsr = 0;
  }

  if (st.mode != 2) {
    const uint32_t ring_base_s = (uint32_t)__cvta_generic_to_shared(smem + warp * RING);
    const uint32_t ring_lane_s = ring_base_s + lane * 16;
    // windows this warp may touch: up to the end of the padded buffer (32-bit counters keep the loop lean)
    const uint64_t avail64 = (p.buf_len - rstart) / WIN;
    const uint32_t n_avail = avail64 > 0xFFFFFFF0ull ? 0xFFFFFFF0u : (uint32_t)avail64;
    const uint32_t seek_limit = (uint32_t)((rend - rstart + WIN - 1) / WIN);  // no owned line can start later
    const uint8_t *gsrc = p.in + rstart + lane * 16;
    uint32_t issue_off = 0;  // ring offset of the next pair of windows
    // one commit group per 1 KiB pair; the buffer carries 8 KiB of slack, so the prefetch needs no bounds test
    auto issue_pair = [&]() {
      const uint32_t d = ring_lane_s + issue_off;
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(d), "l"(gsrc));
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(d + WIN), "l"(gsrc + WIN));
      asm volatile("cp.async.commit_group;\n" ::);
      gsrc += 2 * WIN;
      issue_off = (issue_off + 2 * WIN) & (RING - 1);
    };
#pragma unroll
    for (int k = 0; k < PF_PAIRS; k++) issue_pair();
    // One loop iteration = one 1 KiB pair of windows.  Pairs that are all-reference (the bulk of real
    // data) cost one 9-compare vote; anything else falls through to the per-window dispatcher.
    uint32_t stage_off = 0;
    bool done = false;
    // the vector tiers apply while the warp is inside a line's sample zone with a known field phase; only the
    // general window changes that, so the test is kept as one flag
    bool fast = HAS_SAMPLES && st.mode == 1 && st.col >= 9 && (uint32_t)st.fsr < 4u;
    for (uint32_t it = 0; it + 2 < n_avail && !done; it += 2, stage_off = (stage_off + 2 * WIN) & (RING - 1)) {
      issue_pair();
      asm volatile("cp.async.wait_group %0;\n" ::"n"(PF_PAIRS - 1));  // windows it .. it+3 have landed
      __syncwarp();
      int hint = 0;  // 1: window A was regular and is done, B is known not to be; 2: A is known not to be regular
      if (fast) {
        const uint32_t rp = st.refpat;
        const uint32_t sh = (uint32_t)st.fsr * 8u;
        const uint32_t rot = __funnelshift_l(rp, rp, sh);  // the pattern as the unaligned raw words see it
        uint4 va, vb;
        uint32_t w4b;
        bool allref;
        // T1 x2: every byte of both windows (and the 4 bytes after them) repeats the reference genotype.
        // All-reference pairs come in streaks (most of real data): the streak is a loop of its own, nothing of the
        // warp's state but the column and allele counters moves.  The vote also orders these shared-memory reads
        // before the stages are refilled.
        for (;;) {
          const uint32_t so_b = (stage_off + WIN) & (RING - 1);
          va = lds128(ring_lane_s + stage_off);
          vb = lds128(ring_lane_s + so_b);
          w4b = lds32(ring_base_s + ((so_b + lane * 16 + 16) & (RING - 1)));
          const uint32_t diff = (va.x ^ rot) | (va.y ^ rot) | (va.z ^ rot) | (va.w ^ rot) | (vb.x ^ rot) | (vb.y ^ rot) |
                                (vb.z ^ rot) | (vb.w ^ rot) | (w4b ^ rot);
          allref = __all_sync(FULL, diff == 0);
          if (!allref) break;
          st.a.an_uni += 512; st.col += 256;
          if (!(it + 4 < n_avail)) break;  // the next pair would be the last the loop takes: leave it to the loop
          it += 2; stage_off = (stage_off + 2 * WIN) & (RING - 1);
          issue_pair();
          asm volatile("cp.async.wait_group %0;\n" ::"n"(PF_PAIRS - 1));
          __syncwarp();
        }
        if (allref) continue;
        // T2 x2: both windows regular -> one ordered compaction for the 256 fields
        const uint32_t w4a = lds32(ring_base_s + ((stage_off + lane * 16 + 16) & (RING - 1)));
        const uint32_t ta[4] = {__funnelshift_r(va.x, va.y, sh) ^ rp, __funnelshift_r(va.y, va.z, sh) ^ rp,
                                __funnelshift_r(va.z, va.w, sh) ^ rp, __funnelshift_r(va.w, w4a, sh) ^ rp};
        const uint32_t tb[4] = {__funnelshift_r(vb.x, vb.y, sh) ^ rp, __funnelshift_r(vb.y, vb.z, sh) ^ rp,
                                __funnelshift_r(vb.z, vb.w, sh) ^ rp, __funnelshift_r(vb.w, w4b, sh) ^ rp};
        uint32_t bad = bad_digits8(ta, tb), bad_a = 0;
        bool dots = false;
        if (!__all_sync(FULL, bad == 0)) {
          bad_a = bad_digits_or_dots4(ta, 0xFFFFFFFFu);
          bad = bad_a | bad_digits_or_dots4(tb, 0xFFFFFFFFu);
          dots = true;
        }
        if (__all_sync(FULL, bad == 0)) {
          st.a.an_uni += 512;
          classify_push_pair(p, st, my_events, ta, tb, (int)(st.col - 9) + lane * 4, dots, lane);
          st.col += 256;
          __syncwarp();
          continue;
        }
        // Not regular as a pair (a line ends in it, typically).  What the exact test said about window A spares
        // the per-window dispatcher below its own T1/T2 attempts.
        if (__all_sync(FULL, bad_a == 0)) {
          st.a.an_uni += 256;
          classify_push_words4(p, st, my_events, ta, (int)(st.col - 9) + lane * 4, true, lane);
          st.col += 128;
          hint = 1;
        } else {
          hint = 2;
        }
      }
#pragma unroll 1
      for (int h = 0; h < 2; h++) {
        if (hint == 1 && h == 0) continue;
        const uint32_t wi = it + h;
        const uint32_t so = (stage_off + h * WIN) & (RING - 1);
        if (st.mode == 0 && wi >= seek_limit) { done = true; break; }  // no line starts in this range
        const uint4 v = lds128(ring_lane_s + so);
        if (st.mode == 0) {
          // Seeking the first line that starts in this range (half a line on average, most of a range at biobank
          // width): only a newline matters.  Exact zero-byte test on v ^ '\n', no mask compression.
          const uint32_t K = 0x7F7F7F7Fu;
          const uint32_t a = v.x ^ 0x0A0A0A0Au, b = v.y ^ 0x0A0A0A0Au, c = v.z ^ 0x0A0A0A0Au, d = v.w ^ 0x0A0A0A0Au;
          const uint32_t z = ~((((a & K) + K) | a) & (((b & K) + K) | b) & (((c & K) + K) | c) & (((d & K) + K) | d)) & ~K;
          if (!__any_sync(FULL, z != 0)) continue;
        }
        if (fast && hint != 2 - h) {
          const uint32_t w4 = lds32(ring_base_s + ((so + lane * 16 + 16) & (RING - 1)));
          const uint32_t sh = (uint32_t)st.fsr * 8u;
          const uint32_t rp = st.refpat;
          const uint32_t t[4] = {__funnelshift_r(v.x, v.y, sh) ^ rp, __funnelshift_r(v.y, v.z, sh) ^ rp,
                                 __funnelshift_r(v.z, v.w, sh) ^ rp, __funnelshift_r(v.w, w4, sh) ^ rp};
          if (__all_sync(FULL, (t[0] | t[1] | t[2] | t[3]) == 0)) {  // T1
            st.a.an_uni += 256; st.col += 128;
            continue;
          }
          // T2: separator and tab bytes unchanged, allele bytes in [0-9] (or '.', checked only if needed)
          uint32_t bad = bad_digits4(t, 0xFFFFFFFFu);
          bool dots = false;
          if (!__all_sync(FULL, bad == 0)) {
            bad = bad_digits_or_dots4(t, 0xFFFFFFFFu);
            dots = true;
          }
          if (__all_sync(FULL, bad == 0)) {
            st.a.an_uni += 256;
            classify_push_words4(p, st, my_events, t, (int)(st.col - 9) + lane * 4, dots, lane);
            st.col += 128;
            continue;
          }
        }
        const uint64_t pos = rstart + (uint64_t)wi * WIN;
        scan_window_general<HAS_SAMPLES>(p, st, ring_base_s, so, v, pos, rend, lane, my_recs, my_events);
        if (st.mode == 2) { done = true; break; }
        fast = HAS_SAMPLES && st.mode == 1 && st.col >= 9 && (uint32_t)st.fsr < 4u;
      }
      __syncwarp();  // everyone is done with these stages before they are refilled
    }
  }
  asm volatile("cp.async.wait_group 0;\n" ::);
  if (lane == 0) {
    p.range_nrec[rl] = st.nrec < p.slots_per_range ? st.nrec : p.slots_per_range;  // overflow is flagged
    p.range_nlines[rl] = st.nlines;
  }
}

}  // namespace bvcf
