// bvcf_rows.cuh -- north-star kernels (2)+(3b): what the per-record code shares.
//
//   bvcf_line_stats_kernel      records whose genotype summary is not complete in the scan kernel's LineRec (ALT
//   bvcf_line_stats_big_kernel  numbers other than 1, complex GTs, variable-width names): het/hom/missing counts,
//                               ac, an and list byte lengths for ALT numbers 1..3 from the quad events with nibble
//                               masks (main.go:1042-1194); lane per record, CTA per record with a long event list
//   AlleleGen / gen_next        getAlleles' decision tree as a resumable generator -- ACTG QC, multiallelic split,
//                               MNP decomposition, padding trim + left-normalisation, site type (main.go:723-1038)
//   bvcf_names_big_kernel       warp per queued row, any name widths (bvcf_names.cuh takes fixed-size items)
//
// The rows themselves are composed and written by bvcf_tile_kernel (bvcf_tile.cuh).  Rows of ALT #1..3 use the
// LineRec / LineStats summaries; higher ALT numbers are reduced by the record's own thread straight from the event
// list.
#pragma once
#include "bvcf_common.cuh"
#include "bvcf_text.cuh"

namespace bvcf {

constexpr int NAMES_WARPS = 2;   // small CTAs: rows differ wildly in size, a finished warp must not pin the others' slots
constexpr int FILT_SMEM = 1024;      // FILTER table bytes kept in shared memory

// genotype summary of one (record, ALT number)
struct GtStats {
  uint32_t n_het, n_hom, n_miss, ac, an;
  uint32_t het_bytes, hom_bytes, miss_bytes;  // sum of the sample-name lengths per class
};

// warp-reduced summary of one record for ALT numbers 1..3 (99.99 % of real rows)
constexpr int STAT_ALLELES = 3;
struct __align__(16) LineStats {
  uint32_t n_miss, an, miss_bytes, pad;
  uint32_t n_het[STAT_ALLELES], n_hom[STAT_ALLELES], ac[STAT_ALLELES], het_bytes[STAT_ALLELES], hom_bytes[STAT_ALLELES];
  uint32_t pad2;
};

// one emitted row whose sample-name lists (and dosage row) are left to the names kernels: rows of records with
// more than SMALL_EVENTS event words.  bvcf_tile_kernel appends them to a work list (ordinary rows from the front
// of the array, rows beyond NamesParams::long_words event words from its end).
struct __align__(16) RowDesc {
  uint32_t line;        // record index in the dense line table
  uint32_t allele;      // ALT number (altIdx + 1)
  unsigned long long het_dst, hom_dst, miss_dst;  // absolute byte offsets of the three lists in the output
  uint32_t n_het, n_hom, n_miss;                  // list lengths (names)
  uint32_t row;                                   // row number within the sub-chunk (its dosage row)
};

// diagnostics (main.go:730-986 log.Printf sites): DIAG_WORDS words each -- line_lo, line_hi, alt_no, code, and the
// byte offset of the line in the input region (the host reads CHROM and POS there for the log text)
constexpr uint32_t DIAG_WORDS = 6;
struct DiagSink {
  uint32_t *diags;
  uint32_t cap;
  RunCounters *ctr;
  unsigned long long line_start;   // set per record by the caller
};

// CHROM and POS ("CHROM\tPOS") of the lines of a chunk's diagnostics, gathered on the device for the host's log lines
// when the chunk's text exists only there (bgzf input).  An entry ends before the line's second tab; a line without
// one in its first DIAG_FIELDS_MAX bytes gives an empty entry.
constexpr uint32_t DIAG_FIELDS_MAX = 4096;
__device__ __forceinline__ uint32_t diag_fields_len(const uint8_t *in, unsigned long long len, unsigned long long st) {
  const unsigned long long lim = len < st + DIAG_FIELDS_MAX ? len : st + DIAG_FIELDS_MAX;
  int tabs = 0;
  for (unsigned long long p = st; p < lim; p++) {
    const uint8_t c = in[p];
    if (c == '\n') break;
    if (c == '\t' && ++tabs == 2) return (uint32_t)(p - st);
  }
  return 0;
}
// one CTA: every entry's length, exclusive prefix sums into off[0 .. n] (1,024 entries per step)
__global__ void __launch_bounds__(1024) bvcf_diag_fields_len_kernel(const uint8_t *in, unsigned long long len,
                                                                   const unsigned long long *starts, uint32_t n,
                                                                   unsigned long long *off) {
  __shared__ unsigned long long s_warp[32], s_base;
  const int t = threadIdx.x, lane = t & 31, wid = t >> 5;
  if (t == 0) s_base = 0;
  __syncthreads();
  for (uint32_t b = 0; b < n; b += 1024) {
    const uint32_t i = b + (uint32_t)t;
    const unsigned long long l = i < n ? diag_fields_len(in, len, starts[i]) : 0ull;
    unsigned long long v = l;  // inclusive scan: warp, then warp totals
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const unsigned long long u = __shfl_up_sync(FULL, v, d);
      if (lane >= d) v += u;
    }
    if (lane == 31) s_warp[wid] = v;
    __syncthreads();
    if (wid == 0) {
      unsigned long long w = s_warp[lane];
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const unsigned long long u = __shfl_up_sync(FULL, w, d);
        if (lane >= d) w += u;
      }
      s_warp[lane] = w;
    }
    __syncthreads();
    if (i < n) off[i] = s_base + (wid ? s_warp[wid - 1] : 0ull) + v - l;
    __syncthreads();
    if (t == 0) s_base += s_warp[31];
    __syncthreads();
  }
  if (t == 0) off[n] = s_base;
}
// warp per entry: the bytes to out + off[e]
__global__ void bvcf_diag_fields_copy_kernel(const uint8_t *in, const unsigned long long *starts, const unsigned long long *off,
                                             uint32_t n, uint8_t *out) {
  const uint32_t lane = threadIdx.x & 31, warps = (gridDim.x * blockDim.x) >> 5;
  for (uint32_t e = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; e < n; e += warps) {
    const unsigned long long o = off[e], m = off[e + 1] - o;
    const uint8_t *src = in + starts[e];
    for (uint32_t k = lane; k < m; k += 32) out[o + k] = src[k];
  }
}

// site types (bystro-utils parse.Snp/Ins/Del/Mnp/Multi)
enum { T_SNP = 0, T_INS = 1, T_DEL = 2, T_MNP = 3, T_MULTI = 4 };
__device__ __constant__ char TYPE_TXT[5][13] = {"SNP", "INS", "DEL", "MNP", "MULTIALLELIC"};
__device__ __constant__ int TYPE_LEN[5] = {3, 3, 3, 3, 12};

__device__ __forceinline__ bool is_acgt(uint8_t c) { return c == 'A' || c == 'C' || c == 'G' || c == 'T'; }

// parse.GetTrTv (main.go:605): '1' transition, '2' transversion (single-base alt only)
__device__ __forceinline__ uint8_t trtv_char(uint8_t r, uint8_t a) {
  const bool tr = (r == 'A' && a == 'G') || (r == 'G' && a == 'A') || (r == 'C' && a == 'T') || (r == 'T' && a == 'C');
  return tr ? '1' : '2';
}

__device__ __forceinline__ uint32_t name_len(const DevCfg &c, uint32_t s) {
  return c.name_fixed_w > 0 ? (uint32_t)c.name_fixed_w : c.name_off[s + 1] - c.name_off[s];
}
__device__ __forceinline__ const uint8_t *name_ptr(const DevCfg &c, uint32_t s) {
  return c.names + (c.name_fixed_w > 0 ? (size_t)s * c.name_fixed_w : (size_t)c.name_off[s]);
}

// Events are quads (bvcf_common.cuh); consumers walk the "virtual slots" v = 4 * quad + j of a record:
// slot_load returns the slot word of slot v (EV_OFFSET_TAG when empty / out of range) and, for a complex
// sample, the byte offset of its field.
__device__ __forceinline__ uint32_t slot_load(const uint32_t *ev, uint32_t v, uint32_t n_words, uint32_t &off) {
  const uint32_t q = v >> 2;
  off = 0;
  if (2 * q + 1 >= n_words) return EV_OFFSET_TAG;
  const uint2 e = *reinterpret_cast<const uint2 *>(ev + 2 * q);
  off = e.y;
  return ev_slot_word(e.x, e.y, (int)(v & 3u));
}

// classify one slot word for allele number a; returns class 0..3 (none/het/hom/missing) and gt/alt.
// Complex samples re-parse the field at `off` with the general GT grammar.
__device__ __forceinline__ int classify_word(uint32_t w, uint32_t off, const uint8_t *L,
                                             uint32_t content_len, uint32_t a, uint32_t &samp, uint32_t &gt_extra,
                                             uint32_t &alt) {
  gt_extra = 0; alt = 0; samp = 0;
  if (w & EV_OFFSET_TAG) return 0;
  samp = w & EV_SAMPLE_MASK;
  if (w & EV_COMPLEX) {
    uint32_t gt;
    const int cls = classify_gt_general(L + off, content_len > off ? content_len - off : 0, a, gt, alt);
    gt_extra = gt;  // the scan kernel left this sample out of `an`
    return cls;
  }
  const uint32_t c1 = (w >> 20) & 31, c2 = (w >> 25) & 31;
  if (c1 == EV_CODE_MISSING) return 3;
  alt = (c1 == a) + (c2 == a);   // codes are 0..9: a >= 10 never matches here
  const uint32_t gt = c2 == EV_CODE_ABSENT ? 1 : 2;
  return alt == 0 ? 0 : (alt == gt ? 2 : 1);
}
// slot v of a record's events
__device__ __forceinline__ int classify_event(const uint32_t *ev, uint32_t v, uint32_t n_words, const uint8_t *L,
                                              uint32_t content_len, uint32_t a, uint32_t &samp, uint32_t &gt_extra,
                                              uint32_t &alt, bool &is_ev) {
  uint32_t off;
  const uint32_t w = slot_load(ev, v, n_words, off);
  is_ev = !(w & EV_OFFSET_TAG);
  return classify_word(w, off, L, content_len, a, samp, gt_extra, alt);
}

// ---- nibble-parallel classification of a quad event ---------------------------------------------------
__device__ __forceinline__ uint32_t nib_eq(uint32_t x, uint32_t pat) {  // bit 3 of every nibble of x equal to pat's
  const uint32_t y = x ^ pat;
  return ~(((y & 0x77777777u) + 0x77777777u) | y) & 0x88888888u;
}

// het / hom / missing slots of one quad for allele number a, as nibble flags (bit 4j+3 = sample base+j).
// `simple`: the record only carries alleles 0 / 1 / '.' / absent and a == 1 (LineRec.flags bit 0 clear).
__device__ __forceinline__ void quad_masks(uint32_t h, uint32_t pl, uint32_t a, bool simple, const uint8_t *L,
                                           uint32_t content_len, bool valid, uint32_t &mh, uint32_t &mo, uint32_t &mm) {
  mh = mo = mm = 0;
  if (!valid) return;
  uint32_t one1, one2, dot, hap;
  if (simple) {  // nibbles are 0, 1, 0xE or 0xF: two bit planes tell them apart
    const uint32_t b0 = pl << 3, b3 = pl;
    const uint32_t one = b0 & ~b3 & 0x88888888u, dt = b3 & ~b0 & 0x88888888u;
    one1 = one & 0x8888u; one2 = one >> 16;
    dot = dt | (dt >> 16);
    hap = (b3 & b0 & 0x88888888u) >> 16;
  } else {
    if (h & EV_COMPLEX) {
      uint32_t gt, alt;
      const int cls = classify_gt_general(L + pl, content_len > pl ? content_len - pl : 0, a, gt, alt);
      if (cls == 1) mh = 8u; else if (cls == 2) mo = 8u; else if (cls == 3) mm = 8u;
      return;
    }
    const uint32_t eq = a <= 9 ? nib_eq(pl, a * 0x11111111u) : 0u;
    const uint32_t dt = nib_eq(pl, 0xEEEEEEEEu);
    one1 = eq & 0x8888u; one2 = eq >> 16;
    dot = dt | (dt >> 16);
    hap = nib_eq(pl, 0xFFFFFFFFu) >> 16;
  }
  mm = dot & 0x8888u;
  mo = one1 & (one2 | hap) & ~mm;
  mh = (one1 ^ one2) & ~hap & ~mm & 0x8888u;
}

// ---- warp per record: ALT #1 summary ---------------------------------------------------------------
struct StatsParams {
  const uint8_t *in;
  DevCfg cfg;
  const LineRec *lines;
  const uint32_t *events;
  LineStats *stats;
  RunCounters *ctr;
  uint32_t *big_recs;        // work list: records reduced by a whole warp (bvcf_line_stats_big_kernel)
};

// per-thread partial genotype summary of a record for ALT numbers 1..STAT_ALLELES
struct StatAcc {
  uint32_t n_miss, an_x, mb;
  uint32_t n_het[STAT_ALLELES], n_hom[STAT_ALLELES], ac[STAT_ALLELES], hb[STAT_ALLELES], ob[STAT_ALLELES];
};
__device__ __forceinline__ void stat_zero(StatAcc &s) {
  s.n_miss = s.an_x = s.mb = 0;
#pragma unroll
  for (int a = 0; a < STAT_ALLELES; a++) s.n_het[a] = s.n_hom[a] = s.ac[a] = s.hb[a] = s.ob[a] = 0;
}
// one quad event into the summary: nibble masks per allele number, the general GT grammar for complex samples
// (main.go:1126-1190), name lengths only when the names are not all one width
__device__ __forceinline__ void stat_quad(StatAcc &s, const DevCfg &cfg, bool fixed, uint2 e, const uint8_t *L, uint32_t content_len) {
  const uint32_t s0 = (e.x & EV_SAMPLE_MASK) - EV_BASE_BIAS;
  if (e.x & EV_COMPLEX) {
    const uint32_t nl = fixed ? 0u : name_len(cfg, s0);
#pragma unroll
    for (int a = 0; a < STAT_ALLELES; a++) {
      uint32_t gt, alt;
      const int cls = classify_gt_general(L + e.y, content_len > e.y ? content_len - e.y : 0, a + 1, gt, alt);
      s.ac[a] += alt;
      if (cls == 1) { s.n_het[a]++; s.hb[a] += nl; } else if (cls == 2) { s.n_hom[a]++; s.ob[a] += nl; }
      if (a == 0) { s.an_x += gt; if (cls == 3) { s.n_miss++; s.mb += nl; } }
    }
    return;
  }
  const uint32_t dt = nib_eq(e.y, 0xEEEEEEEEu);
  const uint32_t ms = (dt | (dt >> 16)) & 0x8888u;             // samples with a '.' token
  const uint32_t gone = ((ms | (ms << 16)) >> 3) * 15u;        // both nibbles of those samples
  s.n_miss += __popc(ms);
  uint32_t mh[STAT_ALLELES], mo[STAT_ALLELES];
#pragma unroll
  for (int a = 0; a < STAT_ALLELES; a++) {
    uint32_t mm;
    quad_masks(e.x, e.y, a + 1, false, L, content_len, true, mh[a], mo[a], mm);
    s.n_het[a] += __popc(mh[a]); s.n_hom[a] += __popc(mo[a]);
    s.ac[a] += __popc(nib_eq(e.y, (uint32_t)(a + 1) * 0x11111111u) & ~gone);
  }
  if (!fixed) {
    uint32_t any = ms;
#pragma unroll
    for (int a = 0; a < STAT_ALLELES; a++) any |= mh[a] | mo[a];
    while (any) {  // at most four samples
      const uint32_t bit = any & (0u - any);
      any &= any - 1;
      const uint32_t nl = name_len(cfg, s0 + ((uint32_t)(__ffs(bit) - 1) >> 2));
      if (ms & bit) s.mb += nl;
#pragma unroll
      for (int a = 0; a < STAT_ALLELES; a++) {
        if (mh[a] & bit) s.hb[a] += nl; else if (mo[a] & bit) s.ob[a] += nl;
      }
    }
  }
}

constexpr uint32_t SMALL_EVENTS = 12;  // records with at most this many event words are reduced by one lane

// Hybrid granularity: a warp takes 32 consecutive records.  Each lane reduces its own record when it has
// few events (most of real data: singletons and rare variants); records with long event lists are queued for
// the CTA-per-record kernel.
__global__ void __launch_bounds__(256) bvcf_line_stats_kernel(const StatsParams p) {
  const DevCfg &cfg = p.cfg;
  const int lane = threadIdx.x & 31;
  if (p.ctr->ev_overflow | p.ctr->slot_overflow) return;  // the host grows the scratch and re-runs the chunk
  const uint32_t n_rec = p.ctr->chunk_records;
  const uint32_t total_warps = gridDim.x * (blockDim.x >> 5);
  const bool fixed = cfg.name_fixed_w > 0;
  for (uint32_t lb = (blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * 32; lb < n_rec; lb += total_warps * 32) {
    const uint32_t li = lb + lane;
    const bool valid = li < n_rec;
    LineRec rec;
    rec.start = 0; rec.len = 0; rec.an = 0; rec.ev_start = 0; rec.ev_count = 0; rec.flags = 0;
    if (valid) rec = p.lines[li];
    // records whose inline summary (scan kernel) is complete need nothing here
    const bool needed = valid && (!fixed || (rec.flags & 1));
    const bool small = needed && rec.ev_count <= SMALL_EVENTS;
    if (small) {  // ---- lane-serial ----
      const uint32_t content_len = rec.len >= (uint32_t)cfg.eol_width ? rec.len - (uint32_t)cfg.eol_width : 0;
      const uint32_t *ev = p.events + rec.ev_start;
      StatAcc t;
      stat_zero(t);
      for (uint32_t q = 0; 2 * q + 1 < rec.ev_count; q++)
        stat_quad(t, cfg, fixed, *reinterpret_cast<const uint2 *>(ev + 2 * q), p.in + rec.start, content_len);
      LineStats s;
      s.n_miss = t.n_miss; s.an = rec.an + t.an_x; s.pad = 0; s.pad2 = 0;
      s.miss_bytes = fixed ? t.n_miss * cfg.name_fixed_w : t.mb;
#pragma unroll
      for (int a = 0; a < STAT_ALLELES; a++) {
        s.n_het[a] = t.n_het[a]; s.n_hom[a] = t.n_hom[a]; s.ac[a] = t.ac[a];
        s.het_bytes[a] = fixed ? t.n_het[a] * cfg.name_fixed_w : t.hb[a];
        s.hom_bytes[a] = fixed ? t.n_hom[a] * cfg.name_fixed_w : t.ob[a];
      }
      p.stats[li] = s;
    }
    // ---- the long ones go to the work list of the CTA-per-record kernel (one atomic per warp) ----
    const uint32_t big = __ballot_sync(FULL, needed && !small);
    if (big) {
      uint32_t base = 0;
      if (lane == 0) base = atomicAdd(&p.ctr->n_big_recs, (unsigned int)__popc(big));
      base = __shfl_sync(FULL, base, 0);
      if (needed && !small) p.big_recs[base + __popc(big & ((1u << lane) - 1u))] = li;
    }
  }
}

// CTA per record: the records the hybrid kernel queued (long event lists: up to 50,000 quads at biobank width);
// a thread takes every 256th quad, REDUX per warp, shared-memory atomics across the warps
__global__ void __launch_bounds__(256) bvcf_line_stats_big_kernel(const StatsParams p) {
  __shared__ uint32_t s_wi;
  __shared__ uint32_t s_acc[3 + 5 * STAT_ALLELES];
  const DevCfg &cfg = p.cfg;
  const int lane = threadIdx.x & 31;
  if (p.ctr->ev_overflow | p.ctr->slot_overflow) return;
  const uint32_t n_big = p.ctr->n_big_recs;
  const bool fixed = cfg.name_fixed_w > 0;
  for (;;) {  // CTAs take the next queued record from a shared cursor
    __syncthreads();
    if (threadIdx.x == 0) s_wi = atomicAdd(&p.ctr->big_rec_cursor, 1u);
    if (threadIdx.x < 3 + 5 * STAT_ALLELES) s_acc[threadIdx.x] = 0;
    __syncthreads();
    const uint32_t wi = s_wi;
    if (wi >= n_big) break;
    const uint32_t li = p.big_recs[wi];
    const LineRec rec = p.lines[li];
    const uint32_t content_len = rec.len >= (uint32_t)cfg.eol_width ? rec.len - (uint32_t)cfg.eol_width : 0;
    const uint32_t *ev = p.events + rec.ev_start;
    const uint8_t *L = p.in + rec.start;
    const uint32_t nq = rec.ev_count >> 1;
    StatAcc t;
    stat_zero(t);
    for (uint32_t q = threadIdx.x; q < nq; q += blockDim.x)
      stat_quad(t, cfg, fixed, *reinterpret_cast<const uint2 *>(ev + 2 * q), L, content_len);
    // warp totals -> shared memory
    const uint32_t w_miss = __reduce_add_sync(FULL, t.n_miss), w_an = __reduce_add_sync(FULL, t.an_x), w_mb = __reduce_add_sync(FULL, t.mb);
    uint32_t w[5 * STAT_ALLELES];
#pragma unroll
    for (int a = 0; a < STAT_ALLELES; a++) {
      w[5 * a] = __reduce_add_sync(FULL, t.n_het[a]); w[5 * a + 1] = __reduce_add_sync(FULL, t.n_hom[a]);
      w[5 * a + 2] = __reduce_add_sync(FULL, t.ac[a]); w[5 * a + 3] = __reduce_add_sync(FULL, t.hb[a]);
      w[5 * a + 4] = __reduce_add_sync(FULL, t.ob[a]);
    }
    if (lane == 0) {
      atomicAdd(&s_acc[0], w_miss); atomicAdd(&s_acc[1], w_an); atomicAdd(&s_acc[2], w_mb);
#pragma unroll
      for (int k = 0; k < 5 * STAT_ALLELES; k++) atomicAdd(&s_acc[3 + k], w[k]);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      LineStats s;
      s.n_miss = s_acc[0]; s.pad = 0; s.pad2 = 0;
      s.an = rec.an + s_acc[1];
      s.miss_bytes = fixed ? s.n_miss * cfg.name_fixed_w : s_acc[2];
#pragma unroll
      for (int a = 0; a < STAT_ALLELES; a++) {
        s.n_het[a] = s_acc[3 + 5 * a]; s.n_hom[a] = s_acc[4 + 5 * a];
        s.ac[a] = s_acc[5 + 5 * a];
        s.het_bytes[a] = fixed ? s.n_het[a] * cfg.name_fixed_w : s_acc[6 + 5 * a];
        s.hom_bytes[a] = fixed ? s.n_hom[a] * cfg.name_fixed_w : s_acc[7 + 5 * a];
      }
      p.stats[li] = s;
    }
  }
}

// the record's own thread reduces the events for ALT numbers beyond STAT_ALLELES
__device__ __noinline__ GtStats reduce_events_thread(const DevCfg &cfg, const LineRec &rec, const uint32_t *ev,
                                                     const uint8_t *L, uint32_t content_len, uint32_t a) {
  GtStats s;
  s.n_het = s.n_hom = s.n_miss = s.ac = 0; s.an = rec.an;
  s.het_bytes = s.hom_bytes = s.miss_bytes = 0;
  for (uint32_t k = 0; k < 2 * rec.ev_count; k++) {
    uint32_t samp, gtx, alt;
    bool is_ev;
    const int cls = classify_event(ev, k, rec.ev_count, L, content_len, a, samp, gtx, alt, is_ev);
    s.ac += alt;
    s.an += gtx;
    if (cls) {
      const uint32_t nl = name_len(cfg, samp);
      if (cls == 1) { s.n_het++; s.het_bytes += nl; }
      else if (cls == 2) { s.n_hom++; s.hom_bytes += nl; }
      else { s.n_miss++; s.miss_bytes += nl; }
    }
  }
  return s;
}


// ---- one output allele of getAlleles ------------------------------------------------------------
struct OutAllele {
  long long pos_val;      // used when !pos_verbatim
  const uint8_t *ins_p;   // kind 1: inserted bases
  int ins_n;
  long long del_n;        // kind 2: negative count
  int alt_idx;            // index in the VCF ALT list
  int kind;               // 0 single base, 1 insertion "+...", 2 deletion "-N"
  uint8_t ref, alt_c;
  bool pos_verbatim;
};

struct LineCtx {
  const uint8_t *L;
  uint32_t content_len;
  const uint8_t *chrom, *pos, *id, *info;
  int chrom_n, pos_n, id_n, info_n;
  int site_type;
  bool multi;
  uint32_t li;
};


__device__ __noinline__ void push_diag(const DiagSink &p, unsigned long long line_no, int alt_no, int code) {
  if (!p.diags) return;
  const uint32_t i = atomicAdd(&p.ctr->n_diags, 1u);
  if (i < p.cap) {
    uint32_t *d = p.diags + (size_t)DIAG_WORDS * i;
    d[0] = (uint32_t)line_no; d[1] = (uint32_t)(line_no >> 32);
    d[2] = (uint32_t)alt_no; d[3] = (uint32_t)code;
    d[4] = (uint32_t)p.line_start; d[5] = (uint32_t)(p.line_start >> 32);
  }
}

// ---- getAlleles (main.go:723-1038) as a generator -----------------------------------------------------
// gen_begin does the whole-line checks (REF == ALT, site type); gen_next yields one output allele per call,
// in the order the reference appends them, so that all lanes of a warp meet at a single emit_row call.
struct AlleleGen {
  const uint8_t *ref, *alt;
  int ref_n, alt_n, tn;
  int ta_off;     // the equal-length allele being decomposed base by base: its offset in ALT
  int s;          // cursor in ALT: start of the next comma-separated allele
  int alt_idx;    // its index in the ALT list
  int mnp_i;      // >= 0: resume the MNP decomposition at this base
  long long ipos;
  bool pos_ok, last, done;
  // REF (up to 8 bases) and ALT (up to 16 characters) held in registers: the loops below walk these fields several
  // times a byte at a time, and every byte from memory was a dependent load the whole warp waited for
  bool cached;
  unsigned long long rw, aw0, aw1;
};
__device__ __forceinline__ uint32_t gen_ref(const AlleleGen &g, int i) {
  return g.cached ? (uint32_t)(g.rw >> (8 * i)) & 0xFFu : (uint32_t)g.ref[i];
}
__device__ __forceinline__ uint32_t gen_alt(const AlleleGen &g, int i) {
  if (!g.cached) return g.alt[i];
  const unsigned long long w = i < 8 ? g.aw0 : g.aw1;
  return (uint32_t)(w >> (8 * (i & 7))) & 0xFFu;
}
template <bool CACHE>
__device__ __forceinline__ void gen_cache(AlleleGen &g) {
  g.cached = CACHE && g.ref_n <= 8 && g.alt_n <= 16;
  g.rw = g.aw0 = g.aw1 = 0;
  if (g.cached) {
    g.rw = ld64_any(g.ref);
    g.aw0 = ld64_any(g.alt);
    if (g.alt_n > 8) g.aw1 = ld64_any(g.alt + 8);
  }
}

// CACHE false: a kernel built for 64 registers has no room for the three words (it spilled, and ran slower)
template <bool CACHE = true>
__device__ __forceinline__ void gen_begin(AlleleGen &g, LineCtx &lc, const DiagSink &p, unsigned long long line_no,
                                          bool diag) {
  gen_cache<CACHE>(g);
  bool same = g.alt_n == g.ref_n;
#pragma unroll 1
  for (int i = 0; same && i < g.alt_n; i++) same = gen_alt(g, i) == gen_ref(g, i);
  if (same) {                                                         // :729
    if (diag) push_diag(p, line_no, 0, 1);
    g.done = true;
    return;
  }
  bool multi = false;                                                 // :777-779, 1012: ALT holds a comma
#pragma unroll 1
  for (int i = 0; i < g.alt_n; i++) multi = multi || gen_alt(g, i) == ',';
  lc.multi = multi;
  lc.site_type = T_MULTI;
  if (!multi) {  // a single allele: type from its shape (main.go:742,764,1018-1037)
    if (g.alt_n == 1) lc.site_type = g.ref_n == 1 ? T_SNP : T_DEL;
    else if (g.ref_n == 1 || g.alt_n > g.ref_n) lc.site_type = T_INS;
    else if (g.alt_n < g.ref_n) lc.site_type = T_DEL;
    else {
      int nd = 0;
#pragma unroll 1
      for (int i = 0; i < g.ref_n; i++) nd += gen_ref(g, i) != gen_alt(g, i);
      lc.site_type = nd > 1 ? T_MNP : T_SNP;
    }
  }
}

__device__ __forceinline__ bool gen_next(AlleleGen &g, OutAllele &oa, const DiagSink &p, unsigned long long line_no,
                                         bool diag) {
  const int ref_n = g.ref_n;
  for (;;) {
    if (g.done) return false;
    if (g.mnp_i >= 0) {                                               // :855-873 one row per differing base
#pragma unroll 1
      for (int i = g.mnp_i; i < ref_n; i++) {
        const uint32_t r = gen_ref(g, i), a = gen_alt(g, g.ta_off + i);
        if (r != a) {
          oa.kind = 0; oa.ref = (uint8_t)r; oa.alt_c = (uint8_t)a; oa.pos_verbatim = false; oa.pos_val = g.ipos + i;
          g.mnp_i = i + 1;
          return true;
        }
      }
      g.mnp_i = -1;
      if (g.last) { g.done = true; return false; }
      continue;
    }
    if (g.alt_n == 1) {                                               // :735 the single one-base ALT
      g.done = true;
      const uint8_t a0 = (uint8_t)gen_alt(g, 0);
      oa.alt_idx = 0;
      if (!is_acgt(a0)) { if (diag) push_diag(p, line_no, 1, 2); return false; }
      if (ref_n == 1) {                                               // :742 SNP, POS text verbatim
        oa.kind = 0; oa.ref = (uint8_t)gen_ref(g, 0); oa.alt_c = a0; oa.pos_verbatim = true;
        return true;
      }
      if (a0 != gen_ref(g, 0)) { if (diag) push_diag(p, line_no, 1, 3); return false; }   // :747
      if (!g.pos_ok) { if (diag) push_diag(p, line_no, 1, 4); return false; }      // :752
      oa.kind = 2; oa.ref = (uint8_t)gen_ref(g, 1); oa.del_n = 1 - (long long)ref_n;               // :764
      oa.pos_verbatim = false; oa.pos_val = g.ipos + 1;
      return true;
    }
    // next comma-separated allele                                    // :774
    const int t0 = g.s;  // its offset in ALT
    int e = t0;
#pragma unroll 1
    while (e < g.alt_n && gen_alt(g, e) != ',') e++;
    const int tn = e - t0;
    const bool last = e >= g.alt_n;
    const int alt_idx = g.alt_idx;
    g.s = e + 1;
    g.alt_idx = alt_idx + 1;
    g.last = last;
    if (last) g.done = true;  // cleared again below when an MNP still has bases to yield
    oa.alt_idx = alt_idx;
    bool valid = tn > 0;                                              // altIsValid :456-474
#pragma unroll 1
    for (int i = 0; valid && i < tn; i++) valid = is_acgt((uint8_t)gen_alt(g, t0 + i));
    if (!valid) { if (diag) push_diag(p, line_no, alt_idx + 1, 2); continue; }
    const uint32_t ta0 = gen_alt(g, t0), r0 = gen_ref(g, 0);
    if (ref_n == 1) {                                                 // :786
      if (tn == 1) {
        oa.kind = 0; oa.ref = (uint8_t)r0; oa.alt_c = (uint8_t)ta0; oa.pos_verbatim = true;
        return true;
      }
      if (ta0 != r0) { if (diag) push_diag(p, line_no, alt_idx + 1, 5); continue; }   // :797
      oa.kind = 1; oa.ref = (uint8_t)r0; oa.ins_p = g.alt + t0 + 1; oa.ins_n = tn - 1; oa.pos_verbatim = true;  // :803
      return true;
    }
    if (!g.pos_ok) {                                                  // :822-830 stop, keep what we have
      if (diag) push_diag(p, line_no, 0, 8);
      g.done = true;
      return false;
    }
    if (tn == 1) {                                                    // :832
      if (ta0 != r0) { if (diag) push_diag(p, line_no, alt_idx + 1, 7); continue; }
      oa.kind = 2; oa.ref = (uint8_t)gen_ref(g, 1); oa.del_n = 1 - (long long)ref_n; oa.pos_verbatim = false;
      oa.pos_val = g.ipos + 1;
      return true;
    }
    if (tn == ref_n) {                                                // :855 MNP / padded SNP
      g.ta_off = t0; g.tn = tn; g.mnp_i = 0; g.done = false;
      continue;
    }
    if (tn > ref_n) {                                                 // :899 insertion with padding
      int r = 0;
#pragma unroll 1
      while (tn + r > 0 && ref_n + r > 1 && gen_alt(g, t0 + tn + r - 1) == gen_ref(g, ref_n + r - 1)) r--;
      const int off = ref_n + r;                                      // :932
      bool pre = true;
#pragma unroll 1
      for (int i = 0; pre && i < off; i++) pre = gen_ref(g, i) == gen_alt(g, t0 + i);
      if (!pre) { if (diag) push_diag(p, line_no, alt_idx + 1, 6); continue; }
      oa.kind = 1; oa.ref = (uint8_t)gen_ref(g, off - 1); oa.ins_p = g.alt + t0 + off; oa.ins_n = tn + r - off;
      oa.pos_verbatim = false; oa.pos_val = g.ipos + off - 1;
      return true;
    }
    {                                                                 // :971 deletion with padding
      int r = 0;
#pragma unroll 1
      while (tn + r > 1 && ref_n + r > 0 && gen_alt(g, t0 + tn + r - 1) == gen_ref(g, ref_n + r - 1)) r--;
      const int off = tn + r;                                         // :984
      bool pre = true;
#pragma unroll 1
      for (int i = 0; pre && i < off; i++) pre = gen_ref(g, i) == gen_alt(g, t0 + i);
      if (!pre) { if (diag) push_diag(p, line_no, alt_idx + 1, 6); continue; }
      oa.kind = 2; oa.ref = (uint8_t)gen_ref(g, off); oa.del_n = -((long long)ref_n + r - off);
      oa.pos_verbatim = false; oa.pos_val = g.ipos + off;
      return true;
    }
  }
}

// ---- warp per row: sample-name lists + dosage row ----------------------------------------------------
struct NamesParams {
  const uint8_t *in;
  DevCfg cfg;
  const LineRec *lines;
  const uint32_t *events;
  // the work lists bvcf_copyout_kernel filled: entries [0, ctr->n_mid_rows) are rows written by a lane each
  // (bvcf_names_mid_kernel), the next ctr->n_big_rows entries rows written by a warp each (bvcf_names_vec_kernel);
  // rows with more than long_words event words sit at the END of the array, entries [row_desc_cap -
  // ctr->n_long_rows, row_desc_cap), for bvcf_names_long_kernel (a CTA per row).  bvcf_names_big_kernel serves all
  // three lists when the names are not fixed-size items.
  const RowDesc *row_desc;
  unsigned long long row_desc_cap;
  uint8_t *out;
  RunCounters *ctr;
  int8_t *dosage;            // zeroed by bvcf_copyout_kernel
  unsigned long long dosage_cap_rows;
  uint32_t long_words;       // 0: no CTA-per-row kernel follows
};

// one row, whole warp: ballot/popc ranks, ordered scatter of the names (and the dosage row)
__device__ __forceinline__ void names_row_warp(const NamesParams &p, const RowDesc &rd, unsigned long long row0,
                                               int lane) {
  const DevCfg &cfg = p.cfg;
  const uint32_t dl = (uint32_t)cfg.delim_len;
  const bool fixed = cfg.name_fixed_w > 0;
  const uint32_t lt = (1u << lane) - 1u;
  {
    const LineRec rec = p.lines[rd.line];
    const uint32_t *ev = p.events + rec.ev_start;
    const uint8_t *L = p.in + rec.start;
    const uint32_t content_len = rec.len >= (uint32_t)cfg.eol_width ? rec.len - (uint32_t)cfg.eol_width : 0;
    const uint32_t a = rd.allele;
    int8_t *drow = nullptr;
    if (cfg.want_dosage && p.dosage && (row0 + rd.row) < p.dosage_cap_rows) {
      drow = p.dosage + (row0 + rd.row) * (unsigned long long)cfg.n_samples;  // zeroed by bvcf_tile_kernel
    }
    uint32_t run_n[3] = {0, 0, 0};
    uint32_t run_b[3] = {0, 0, 0};
    const unsigned long long dsts[3] = {rd.het_dst, rd.hom_dst, rd.miss_dst};
    for (uint32_t base = 0; base < 2 * rec.ev_count; base += 32) {
      uint32_t samp, gtx, alt;
      const uint32_t k = base + lane;
      bool is_ev;
      const int cls = classify_event(ev, k, rec.ev_count, L, content_len, a, samp, gtx, alt, is_ev);
      if (drow && is_ev)
        drow[samp] = cls == 3 ? (int8_t)-1 : (int8_t)(alt > 127 ? 127 : alt);  // main.go:1172-1178
      if (!cfg.want_tsv) continue;
      const uint32_t nl = cls ? name_len(cfg, samp) : 0;
      uint32_t my_off = 0, my_idx = 0;
#pragma unroll
      for (int c = 0; c < 3; c++) {
        const uint32_t bal = __ballot_sync(FULL, cls == c + 1);
        if (bal == 0) continue;
        const uint32_t rank = __popc(bal & lt);
        const uint32_t cnt = __popc(bal);
        if (fixed) {
          if (cls == c + 1) { my_idx = run_n[c] + rank; my_off = my_idx * (cfg.name_fixed_w + dl); }
          run_n[c] += cnt;
        } else {
          const uint32_t v = cls == c + 1 ? nl + dl : 0;
          const uint32_t incl = warp_incl_scan(v, lane);
          if (cls == c + 1) { my_idx = run_n[c] + rank; my_off = run_b[c] + incl - v; }
          run_n[c] += cnt;
          run_b[c] += __shfl_sync(FULL, incl, 31);
        }
      }
      if (cls) {
        // item i occupies [delim if i>0] + name; my_off counts a delimiter per earlier item
        uint8_t *d = p.out + dsts[cls - 1] + my_off;
        if (my_idx > 0)
          for (uint32_t i = 0; i < dl; i++) d[(int)i - (int)dl] = cfg.delim[i];
        const uint8_t *src = name_ptr(cfg, samp);
        for (uint32_t i = 0; i < nl; i++) d[i] = src[i];
      }
    }
  }
}


// 8 bytes to an arbitrarily aligned address with the widest naturally aligned pieces (2-4 stores)
__device__ __forceinline__ void store8_unaligned(uint8_t *d, unsigned long long v) {
  const uint32_t lo = (uint32_t)v, hi = (uint32_t)(v >> 32);
  switch ((uintptr_t)d & 3u) {
    case 0:
      *reinterpret_cast<uint32_t *>(d) = lo;
      *reinterpret_cast<uint32_t *>(d + 4) = hi;
      break;
    case 2:
      *reinterpret_cast<uint16_t *>(d) = (uint16_t)lo;
      *reinterpret_cast<uint32_t *>(d + 2) = (uint32_t)(v >> 16);
      *reinterpret_cast<uint16_t *>(d + 6) = (uint16_t)(hi >> 16);
      break;
    case 1:
      d[0] = (uint8_t)lo;
      *reinterpret_cast<uint16_t *>(d + 1) = (uint16_t)(lo >> 8);
      *reinterpret_cast<uint32_t *>(d + 3) = (uint32_t)(v >> 24);
      d[7] = (uint8_t)(hi >> 24);
      break;
    default:
      d[0] = (uint8_t)lo;
      *reinterpret_cast<uint32_t *>(d + 1) = (uint32_t)(v >> 8);
      *reinterpret_cast<uint16_t *>(d + 5) = (uint16_t)(hi >> 8);
      d[7] = (uint8_t)(hi >> 24);
      break;
  }
}

// one row, one lane: rows whose record has a moderate number of events (up to TileParams::mid_words).  A warp per
// such row spent some 1,000 instructions on a list of a dozen names (a sweep step, three emit calls, 31 idle lanes).
template <bool DOSAGE>
__device__ __forceinline__ void names_row_lane(const NamesParams &p, const RowDesc &rd, const LineRec &rec, int8_t *drow) {
  const DevCfg &cfg = p.cfg;
  const uint32_t *ev = p.events + rec.ev_start;
  const uint8_t *L = p.in + rec.start;
  const uint32_t content_len = rec.len >= (uint32_t)cfg.eol_width ? rec.len - (uint32_t)cfg.eol_width : 0;
  const uint32_t dl = (uint32_t)cfg.delim_len;
  const bool simple = !(rec.flags & 1) && rd.allele == 1;
  // per-class cursors in scalars (a runtime-indexed array would live in local memory)
  uint32_t nh = 0, no = 0, nm = 0, bh = 0, bo = 0, bm = 0;
  for (uint32_t q = 0; 2 * q + 1 < rec.ev_count; q++) {
    const uint2 e = *reinterpret_cast<const uint2 *>(ev + 2 * q);
    uint32_t mh, mo, mm;
    quad_masks(e.x, e.y, rd.allele, simple, L, content_len, true, mh, mo, mm);
    const uint32_t s0 = (e.x & EV_SAMPLE_MASK) - EV_BASE_BIAS;
    uint32_t any = mh | mo | mm;
    while (any) {
      const uint32_t bit = any & (0u - any);
      any &= any - 1;
      const uint32_t samp = s0 + ((uint32_t)(__ffs(bit) - 1) >> 2);
      const bool is_h = (mh & bit) != 0, is_o = (mo & bit) != 0;
      if (DOSAGE && drow) {  // int8 dosage: -1 missing, else min(number of alleles equal to the row's, 127) (main.go:1172-1178)
        int v = -1;
        if (is_h | is_o) {
          if (e.x & EV_COMPLEX) {
            uint32_t gt, alt;
            classify_gt_general(L + e.y, content_len > e.y ? content_len - e.y : 0, rd.allele, gt, alt);
            v = alt > 127 ? 127 : (int)alt;
          } else {
            const uint32_t sh = (uint32_t)(__ffs(bit) - 1) - 3u;  // 4 * slot
            const bool hap = ((e.y >> (16 + sh)) & 0xFu) == EV_NIB_ABSENT;
            v = is_h ? 1 : (hap ? 1 : 2);
          }
        }
        drow[samp] = (int8_t)v;
      }
      const uint32_t rn = is_h ? nh : (is_o ? no : nm), rb = is_h ? bh : (is_o ? bo : bm);
      const unsigned long long dst = is_h ? rd.het_dst : (is_o ? rd.hom_dst : rd.miss_dst);
      const uint32_t tot = is_h ? rd.n_het : (is_o ? rd.n_hom : rd.n_miss);
      uint8_t *d = p.out + dst + rb;
      uint32_t adv = 0;
      if (rn > 0) {
        for (uint32_t i = 0; i < dl; i++) d[i] = cfg.delim[i];
        d += dl; adv = dl;
      }
      const uint32_t nl = name_len(cfg, samp);
      if (cfg.name8) {
        unsigned long long it = cfg.name8[samp];
        if (rn + 1 == tot) it = (it & 0x00FFFFFFFFFFFFFFull) | ((unsigned long long)'\t' << 56);  // after the last name
        store8_unaligned(d, it);
      } else {
        const uint8_t *src = name_ptr(cfg, samp);
        for (uint32_t i = 0; i < nl; i++) d[i] = src[i];
      }
      adv += nl;
      if (is_h) { nh++; bh += adv; } else if (is_o) { no++; bo += adv; } else { nm++; bm += adv; }
    }
  }
}

// lane per row: the mid list (TSV output only)
template <bool DOSAGE>
__global__ void __launch_bounds__(128) bvcf_names_mid_kernel(const NamesParams p) {
  const DevCfg &cfg = p.cfg;
  if (p.ctr->out_overflow | p.ctr->ev_overflow | p.ctr->slot_overflow | p.ctr->row_overflow | p.ctr->scratch_overflow) return;
  const unsigned long long row0 = p.ctr->chunk_row_base;
  const uint32_t n_mid = p.ctr->n_mid_rows;
  for (uint32_t r = blockIdx.x * blockDim.x + threadIdx.x; r < n_mid; r += gridDim.x * blockDim.x) {
    const RowDesc rd = p.row_desc[r];
    const LineRec rec = p.lines[rd.line];
    int8_t *drow = nullptr;
    if (DOSAGE && cfg.want_dosage && p.dosage && (row0 + rd.row) < p.dosage_cap_rows)
      drow = p.dosage + (row0 + rd.row) * (unsigned long long)cfg.n_samples;
    names_row_lane<DOSAGE>(p, rd, rec, drow);
  }
}

// warp per row: the rows bvcf_tile_kernel queued, when the list items are not fixed 8-byte pieces
// (variable-width names or a longer delimiter; otherwise bvcf_names.cuh takes them)
__global__ void __launch_bounds__(NAMES_WARPS * 32) bvcf_names_big_kernel(const NamesParams p) {
  const int lane = threadIdx.x & 31;
  if (p.ctr->out_overflow | p.ctr->ev_overflow | p.ctr->slot_overflow | p.ctr->row_overflow) return;
  const unsigned long long row0 = p.ctr->chunk_row_base;
  const uint32_t n_big = p.ctr->n_mid_rows + p.ctr->n_big_rows, n_long = p.ctr->n_long_rows;
  const uint32_t total_warps = gridDim.x * NAMES_WARPS;
  for (uint32_t wi = blockIdx.x * NAMES_WARPS + (threadIdx.x >> 5); wi < n_big + n_long; wi += total_warps)
    names_row_warp(p, wi < n_big ? p.row_desc[wi] : p.row_desc[p.row_desc_cap - 1 - (wi - n_big)], row0, lane);
}

}  // namespace bvcf
