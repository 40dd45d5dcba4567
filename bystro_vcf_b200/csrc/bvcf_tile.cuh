// bvcf_tile.cuh -- north-star kernels (2)+(4): the per-line fixed-field kernel and the row emitter, generator run ONCE.
//
// Tiles of 32 consecutive records, a warp per tile, one thread per record, no ordering between tiles anywhere:
//   bvcf_compose_kernel   FILTER allow/exclude against a shared-memory table (main.go:447-454), getAlleles
//                         (main.go:723-1038, the generator of bvcf_rows.cuh), genotype summary lookup, ac == 0 skip
//                         (main.go:558), and the TEXT of every row (main.go:586-695) composed with byte stores into a
//                         shared-memory arena: fixed columns, float text, and -- for records with at most
//                         SMALL_EVENTS event words -- the sample-name lists too (main.go:617,639,653), so that such a
//                         row is one contiguous string.  Long lists stay holes.  The tile's arena, row table and
//                         per-record sizes leave as one compact block of a global scratch buffer (coalesced 16-byte
//                         stores) next to the tile's totals: bytes, rows, locus bytes, queued rows.
//   bvcf_tile_{reduce,spine,offsets}_kernel   exclusive scan of the tile totals -> every tile's place in the output,
//                         in the locus buffer and in the RowDesc work lists; advances the run's cursors.
//   bvcf_copyout_kernel   pulls a tile's block back into shared memory and lets every thread copy its rows to the
//                         output with aligned 8-byte stores (funnel-shifted shared-memory words); appends the INFO span
//                         straight from the input line, writes locus strings + the small rows' dosages
//                         (main.go:576-584), queues the rows with holes for the names kernels (bvcf_names.cuh).
//   bvcf_slow_rows_kernel records that did not fit the arena (very long alleles / IDs, dozens of rows per record):
//                         sized by the compose kernel with the stores switched off, written here by one thread each
//                         straight to global memory.
//
// Replaces round 1's bvcf_rows_kernel<SIZE> + 3 prefix kernels + bvcf_rows_kernel<EMIT> + bvcf_names_kernel
// (+ bvcf_rows_list_kernel x2, bvcf_dosage_zero_kernel): that pair ran the generator twice and spent 60 % of its
// instructions in an 8-byte register writer with unaligned global stores.  A single-kernel version with a decoupled
// look-back between the tiles was measured first and dropped: with thousands of tiles in flight every wave waited
// for its slowest tile's compose phase (45 % of the issued instructions were look-back polls).
#pragma once
#include "bvcf_rows.cuh"

namespace bvcf {

constexpr int TILE_THREADS = 32;           // records per tile, one thread each: a tile is a warp's
constexpr int TILE_WARPS = 4;              // warps (independent tiles) per CTA
constexpr uint32_t TILE_ROWS_MAX = 160;    // most staged rows per tile any kernel variant allows; lane l's first row is rows[l]
constexpr uint32_t ROW_NONE = 0xFFFFu;

// one staged row (shared memory, then the tile's scratch block)
struct __align__(16) TRow {
  uint32_t hole_len[3];   // bytes of the het / hom / missing list when it is NOT staged (filled by the names kernels)
  uint16_t hole_pos[3];   // where the hole sits in the staged string (staged bytes before it)
  uint16_t soff;          // arena offset of the staged string: TSV bytes, the locus, then (queued rows) three counts
  uint16_t slen;          // staged TSV bytes
  uint16_t loc_len;       // staged locus bytes
  uint16_t next;          // next row of the same record, ROW_NONE at the end
  uint16_t allele;        // ALT number
  uint16_t flags;         // bit 0: the INFO span and the EOL follow the staged bytes; bit 1: queue a RowDesc
  uint16_t pad;
};
static_assert(sizeof(TRow) == 32, "TRow layout");

// what one record contributes to its tile (scratch block, one per lane)
struct __align__(16) LaneRec {
  unsigned long long bytes;   // TSV bytes of all its rows
  uint32_t rows, loci;        // rows, locus bytes
  uint32_t n_desc;            // RowDesc entries it will queue
  uint16_t first;             // its first staged row (chain through TRow::next)
  uint16_t flags;             // bit 0: slow path (nothing staged, the sizes are still exact); bits 1-2: work list of its queued rows
  uint32_t info_off, info_n;  // INFO span of its line (offset from the line start)
};
static_assert(sizeof(LaneRec) == 32, "LaneRec layout");

// a tile's totals (compose kernel) and where its scratch block is
struct __align__(16) TileAgg {
  unsigned long long bytes;
  unsigned long long scratch_off;     // byte offset of the block in the scratch buffer
  uint32_t rows, loci, n_big, n_long;
  uint32_t arena_used, n_trows;       // block layout: 32 LaneRec, n_trows TRow, arena_used bytes (16-byte padded)
  uint32_t n_mid;
  uint32_t flags;                     // bit 0: dense block -- nothing but the tile's output bytes, in order (sites-only composer)
};
static_assert(sizeof(TileAgg) == 48, "TileAgg layout");
// exclusive prefix of the totals over the tiles before this one (tile offsets kernels)
struct __align__(16) TileBase {
  unsigned long long bytes, loci;
  uint32_t rows, n_big, n_long, n_mid;
};
static_assert(sizeof(TileBase) == 32, "TileBase layout");
// a slow-path record with its place in the outputs (copy-out kernel -> slow rows kernel)
struct __align__(16) SlowRec {
  unsigned long long out_off, loci_off;
  uint32_t li, row, desc, flags;      // flags bit 0: RowDesc slots are available, bits 1-2: work list
};

struct TileParams {
  const uint8_t *in;
  DevCfg cfg;
  const LineRec *lines;        // dense, input order
  const uint32_t *events;      // sub-chunk event buffer
  const LineStats *stats;      // per record, ALT #1..3 (null when there are no samples)
  uint8_t *out;
  unsigned long long out_cap;
  RunCounters *ctr;
  TileAgg *tile_agg;           // per tile
  TileBase *tile_base;         // per tile
  unsigned long long *tile_partial;  // TSCAN_BLOCKS x 5
  uint8_t *scratch;            // tile blocks
  unsigned long long scratch_cap;
  SlowRec *slow;               // slow-path records of the sub-chunk
  uint32_t slow_cap;
  RowDesc *row_desc;           // work list for the names kernels (see RowDesc)
  unsigned long long row_desc_cap;
  // queued rows by the event words of their record: up to mid_words -> the lane-per-row names kernel (entries from
  // the front of row_desc), more than long_words -> the CTA-per-row kernel (entries from the END of row_desc), the
  // rest -> the warp-per-row kernel (entries after the mid ones); 0: no such class
  uint32_t mid_words, long_words;
  // dosage matrix (main.go:576-584)
  int8_t *dosage;              // rows x n_samples
  unsigned long long dosage_cap_rows;
  uint8_t *loci;               // locus strings "chrom:pos:ref:alt", back to back
  unsigned long long loci_cap;
  unsigned long long *loci_off;  // dosage_cap_rows entries: start of row r's locus in `loci`
  DiagSink diag;
};

// staged bytes: no "memory" clobber on purpose -- the arena is only read back after a __syncwarp(), and with the
// clobber every global byte load of a span() had to complete before the next one could even be issued
__device__ __forceinline__ void sts8(uint32_t a, uint32_t v) { asm volatile("st.shared.u8 [%0], %1;\n" ::"r"(a), "r"(v)); }
__device__ __forceinline__ void sts32(uint32_t a, uint32_t v) { asm volatile("st.shared.u32 [%0], %1;\n" ::"r"(a), "r"(v)); }
// up to 7 bytes of v (little-endian) to g, widest naturally aligned pieces first where the address allows
__device__ __forceinline__ void store_head(uint8_t *&g, unsigned long long &v, uint32_t &n, uint32_t &moved) {
  // bytes up to the next 8-byte boundary of g (at most n)
  moved = 0;
  if (((uintptr_t)g & 1u) && n >= 1) { *g = (uint8_t)v; v >>= 8; g += 1; n -= 1; moved += 1; }
  if (((uintptr_t)g & 2u) && n >= 2) { *reinterpret_cast<uint16_t *>(g) = (uint16_t)v; v >>= 16; g += 2; n -= 2; moved += 2; }
  if (((uintptr_t)g & 4u) && n >= 4) { *reinterpret_cast<uint32_t *>(g) = (uint32_t)v; v >>= 32; g += 4; n -= 4; moved += 4; }
}
__device__ __forceinline__ void store_tail(uint8_t *g, unsigned long long v, uint32_t n) {  // n < 8, g 8-byte aligned or n small
  if (n & 4u) { *reinterpret_cast<uint32_t *>(g) = (uint32_t)v; v >>= 32; g += 4; }
  if (n & 2u) { *reinterpret_cast<uint16_t *>(g) = (uint16_t)v; v >>= 16; g += 2; }
  if (n & 1u) *g = (uint8_t)v;
}
__device__ __forceinline__ unsigned long long ldg64_unaligned(const uint8_t *s) { return ld64_any(s); }

// n bytes from global memory (a tile's scratch block, a span of the input line: both padded, so whole words may be
// read) to global memory, any alignments: at most three narrow stores up to the first 8-byte boundary of the
// destination, aligned 8-byte stores of funnel-shifted source words, at most three narrow stores at the end.
__device__ __forceinline__ void copy_g2g(uint8_t *__restrict__ g_, const uint8_t *__restrict__ s_, uint32_t n) {
  if (n == 0) return;
  uint8_t *g = g_;
  const uint8_t *s = s_;
  if ((uintptr_t)g & 7u) {
    unsigned long long v = ldg64_unaligned(s);
    if (n < 8 && (((uintptr_t)g & 7u) + n) <= 8u) {  // the whole piece sits inside one 8-byte word of the destination
      for (uint32_t i = 0; i < n; i++) g[i] = (uint8_t)(v >> (8 * i));
      return;
    }
    uint32_t moved;
    store_head(g, v, n, moved);
    s += moved;
  }
  if (n >= 8) {
    const uint32_t sh = (uint32_t)((uintptr_t)s & 3u) * 8u;
    const uint32_t *__restrict__ wp = reinterpret_cast<const uint32_t *>((uintptr_t)s & ~(uintptr_t)3);
    uint32_t w0 = wp[0];
    // 32 bytes per round, all eight source words in flight before the first store (the source is an L2 round trip
    // away: one word pair per round trip made this loop the copy-out kernel's whole run time)
    while (n >= 32) {
      const uint32_t w1 = wp[1], w2 = wp[2], w3 = wp[3], w4 = wp[4], w5 = wp[5], w6 = wp[6], w7 = wp[7], w8 = wp[8];
      uint2 *gv = reinterpret_cast<uint2 *>(g);
      gv[0] = make_uint2(__funnelshift_r(w0, w1, sh), __funnelshift_r(w1, w2, sh));
      gv[1] = make_uint2(__funnelshift_r(w2, w3, sh), __funnelshift_r(w3, w4, sh));
      gv[2] = make_uint2(__funnelshift_r(w4, w5, sh), __funnelshift_r(w5, w6, sh));
      gv[3] = make_uint2(__funnelshift_r(w6, w7, sh), __funnelshift_r(w7, w8, sh));
      w0 = w8; wp += 8; g += 32; s += 32; n -= 32;
    }
    while (n >= 8) {
      const uint32_t w1 = wp[1], w2 = wp[2];
      *reinterpret_cast<uint2 *>(g) = make_uint2(__funnelshift_r(w0, w1, sh), __funnelshift_r(w1, w2, sh));
      w0 = w2; wp += 2; g += 8; s += 8; n -= 8;
    }
  }
  if (n) store_tail(g, ldg64_unaligned(s), n);
}

// ---- byte sinks of the row composer ---------------------------------------------------------------------
// StageWriter: shared memory while `stg`, a plain byte count otherwise (slow-path records are sized with it).
struct StageWriter {
  static constexpr bool kStage = true;
  uint32_t a;   // shared-memory address of the next byte
  bool stg;
  __device__ __forceinline__ void byte(uint32_t c) { if (stg) sts8(a, c); a++; }
  __device__ __forceinline__ void packed(unsigned long long chars, int len) {  // len <= 8 characters, little-endian
    if (stg) {
      // a rolled loop on purpose: unrolled and inlined at some thirty call sites this was 7,000 instructions of a
      // kernel that stalled on instruction fetch
      uint32_t lo = (uint32_t)chars, hi = (uint32_t)(chars >> 32);
#pragma unroll 1
      for (int k = 0; k < len; k++) { sts8(a + k, lo & 0xFFu); lo = __funnelshift_r(lo, hi, 8); hi >>= 8; }
    }
    a += len;
  }
  // a span of the INPUT (padded: whole words may be read): eight bytes per round trip to memory instead of one
  __device__ __forceinline__ void span(const uint8_t *p, int len) {
    if (stg) {
#pragma unroll 1
      for (int i = 0; i < len; i += 8) {
        const unsigned long long v = ld64_any(p + i);
        uint32_t lo = (uint32_t)v, hi = (uint32_t)(v >> 32);
        const int m = len - i < 8 ? len - i : 8;
#pragma unroll 1
        for (int k = 0; k < m; k++) { sts8(a + i + k, lo & 0xFFu); lo = __funnelshift_r(lo, hi, 8); hi >>= 8; }
      }
    }
    a += len;
  }
  // bytes of the configuration (kernel parameters, constant memory)
  __device__ __forceinline__ void span_const(const uint8_t *p, int len) {
    if (stg) {
#pragma unroll 1
      for (int i = 0; i < len; i++) sts8(a + i, p[i]);
    }
    a += len;
  }
};
// GlobalWriter: the slow path's second pass, byte stores straight to the output (`on` false: the output region
// is too small, the host will re-run the chunk)
struct GlobalWriter {
  static constexpr bool kStage = false;
  uint8_t *g;
  bool on;
  __device__ __forceinline__ void byte(uint32_t c) { if (on) *g = (uint8_t)c; g++; }
  __device__ __forceinline__ void packed(unsigned long long chars, int len) {
    if (on) {
#pragma unroll 1
      for (int k = 0; k < len; k++) g[k] = (uint8_t)(chars >> (8 * k));
    }
    g += len;
  }
  __device__ __forceinline__ void span(const uint8_t *p, int len) {
    if (on) {
#pragma unroll 1
      for (int i = 0; i < len; i++) g[i] = p[i];
    }
    g += len;
  }
  __device__ __forceinline__ void span_const(const uint8_t *p, int len) { span(p, len); }
};
template <class W>
__device__ __noinline__ void w_dec_long(W &w, long long v) {  // more than 16 characters: out of line, it never runs on real data
  uint8_t buf[24];
  const int l2 = itoa_dec(v, buf);
#pragma unroll 1
  for (int i = 0; i < l2; i++) w.byte(buf[i]);
}
template <class W>
__device__ __forceinline__ void w_dec(W &w, long long v) {  // strconv.Itoa
  unsigned long long lo, hi;
  const int len = itoa_pack(v, lo, hi);  // registers, no byte buffer in local memory
  if (len >= 0) {
    w.packed(lo, len < 8 ? len : 8);
    if (len > 8) w.packed(hi, len - 8);
  } else {
    w_dec_long(w, v);
  }
}

// counts below 10,000 (ac, an of most cohorts) without the digit loop of itoa_pack
template <class W>
__device__ __forceinline__ void w_dec_small(W &w, uint32_t v) {
  if (v >= 10000u) { w_dec(w, (long long)v); return; }
  const uint32_t d3 = v / 1000u, r3 = v - d3 * 1000u, d2 = r3 / 100u, r2 = r3 - d2 * 100u, d1 = r2 / 10u, d0 = r2 - d1 * 10u;
  const uint32_t txt = (0x30u + d3) | ((0x30u + d2) << 8) | ((0x30u + d1) << 16) | ((0x30u + d0) << 24);
  const int len = v >= 1000u ? 4 : (v >= 100u ? 3 : (v >= 10u ? 2 : 1));
  w.packed((unsigned long long)(txt >> (8 * (4 - len))), len);
}
// what one record contributes to its tile
struct RecOut {
  unsigned long long bytes;   // TSV bytes of all its rows
  uint32_t rows, loci;        // rows, locus bytes
  uint32_t n_desc;            // RowDesc entries it will queue
  uint32_t first, last;       // its staged rows (chain through TRow::next)
  bool failed;                // slow path: nothing staged, the sizes above are still exact
};
struct TileShared {
  uint32_t arena_s;           // shared-memory address of the arena
  uint32_t arena_cap;         // its size
  uint32_t rows_cap;          // row descriptors
  TRow *rows;
  uint32_t *arena_cur, *rows_cur;
};
// slow-path pass 2: where the record's rows, loci and RowDesc entries go
struct SlowOut {
  unsigned long long row;       // next row number within the sub-chunk
  unsigned long long loci_off;  // next locus byte (absolute in `loci`)
  uint32_t desc;                // next RowDesc ordinal of this record's list
  int cls;                      // 0 mid, 1 big, 2 long (see TileParams::mid_words)
  bool desc_ok;
};

// entry `ord` of work list `cls`: mid rows from the front, big rows after ALL the mid rows of the sub-chunk (their
// count is final once the tile spine kernel has run), long rows from the end
__device__ __forceinline__ void queue_row_desc(const TileParams &p, int cls, uint32_t ord, const RowDesc &rd) {
  const unsigned long long slot = cls == 2 ? p.row_desc_cap - 1ull - ord : (cls == 1 ? (unsigned long long)p.ctr->n_mid_rows + ord : ord);
  p.row_desc[slot] = rd;
}
__device__ __forceinline__ int row_class(const TileParams &p, uint32_t ev_count) {
  if (p.long_words && ev_count > p.long_words) return 2;
  return (p.mid_words && ev_count <= p.mid_words) ? 0 : 1;
}

// the names of a short record's row into the staged lists (main.go:617,639,653 strings.Join): one walk over the
// record's quad events (at most SMALL_EVENTS / 2), header order
// SPEC (everywhere below): the kernel is built for the default flags -- TSV rows, no --keepPos/Id/Info, no dosage
// matrix, 7-character sample names and a one-character delimiter -- and the code of the other cases is not in it
template <bool SPEC>
__device__ __forceinline__ void fill_small_lists(const TileParams &p, const LineRec &rec, const LineCtx &lc, uint32_t a,
                                                 uint32_t la0, uint32_t la1, uint32_t la2) {
  const DevCfg &cfg = p.cfg;
  const uint32_t *ev = p.events + rec.ev_start;
  const bool simple = !(rec.flags & 1) && a == 1;
  const uint32_t dl = SPEC ? 1u : (uint32_t)cfg.delim_len;
  uint32_t nh = 0, no = 0, nm = 0;
  for (uint32_t q = 0; 2 * q + 1 < rec.ev_count; q++) {
    const uint2 e = *reinterpret_cast<const uint2 *>(ev + 2 * q);
    uint32_t mh, mo, mm;
    quad_masks(e.x, e.y, a, simple, lc.L, lc.content_len, true, mh, mo, mm);
    const uint32_t s0 = (e.x & EV_SAMPLE_MASK) - EV_BASE_BIAS;
    uint32_t any = mh | mo | mm;
    while (any) {
      const uint32_t bit = any & (0u - any);
      any &= any - 1;
      const uint32_t samp = s0 + ((uint32_t)(__ffs(bit) - 1) >> 2);
      const bool is_h = (mh & bit) != 0, is_o = (mo & bit) != 0;
      uint32_t d = is_h ? la0 : (is_o ? la1 : la2);
      const uint32_t rn = is_h ? nh : (is_o ? no : nm);
      if (rn > 0) {
        for (uint32_t i = 0; i < dl; i++) sts8(d + i, cfg.delim[i]);
        d += dl;
      }
      const uint32_t nl = SPEC ? 7u : name_len(cfg, samp);
      if (SPEC || cfg.name8) {
        const unsigned long long it = cfg.name8[samp];
#pragma unroll
        for (int i = 0; i < 7; i++) sts8(d + i, (uint32_t)(it >> (8 * i)) & 0xFFu);
      } else {
        const uint8_t *src = name_ptr(cfg, samp);
        for (uint32_t i = 0; i < nl; i++) sts8(d + i, src[i]);
      }
      d += nl;
      if (is_h) { nh++; la0 = d; } else if (is_o) { no++; la1 = d; } else { nm++; la2 = d; }
    }
  }
}

// the int8 dosages of a short record's row (main.go:1172-1178): -1 missing, else min(alleles equal to the row's, 127);
// the row was zeroed by the tile
__device__ __forceinline__ void small_dosage(const TileParams &p, const LineRec &rec, uint32_t a, int8_t *drow) {
  const DevCfg &cfg = p.cfg;
  const uint32_t *ev = p.events + rec.ev_start;
  const uint8_t *L = p.in + rec.start;
  const uint32_t content_len = rec.len >= (uint32_t)cfg.eol_width ? rec.len - (uint32_t)cfg.eol_width : 0;
  const bool simple = !(rec.flags & 1) && a == 1;
  for (uint32_t q = 0; 2 * q + 1 < rec.ev_count; q++) {
    const uint2 e = *reinterpret_cast<const uint2 *>(ev + 2 * q);
    uint32_t mh, mo, mm;
    quad_masks(e.x, e.y, a, simple, L, content_len, true, mh, mo, mm);
    const uint32_t s0 = (e.x & EV_SAMPLE_MASK) - EV_BASE_BIAS;
    uint32_t any = mh | mo | mm;
    while (any) {
      const uint32_t bit = any & (0u - any);
      any &= any - 1;
      const uint32_t samp = s0 + ((uint32_t)(__ffs(bit) - 1) >> 2);
      const bool is_h = (mh & bit) != 0, is_o = (mo & bit) != 0;
      int v = -1;
      if (is_h | is_o) {
        if (e.x & EV_COMPLEX) {
          uint32_t gt, alt;
          classify_gt_general(L + e.y, content_len > e.y ? content_len - e.y : 0, a, gt, alt);
          v = alt > 127 ? 127 : (int)alt;
        } else {
          const uint32_t sh = (uint32_t)(__ffs(bit) - 1) - 3u;  // 4 * slot
          const bool hap = ((e.y >> (16 + sh)) & 0xFu) == EV_NIB_ABSENT;
          v = is_h ? 1 : (hap ? 1 : 2);
        }
      }
      drow[samp] = (int8_t)v;
    }
  }
}

// CountWriter: the length of a text without writing it
struct CountWriter {
  static constexpr bool kStage = true;
  uint32_t a;
  __device__ __forceinline__ void byte(uint32_t) { a++; }
  __device__ __forceinline__ void packed(unsigned long long, int len) { a += len; }
  __device__ __forceinline__ void span(const uint8_t *, int len) { a += len; }
  __device__ __forceinline__ void span_const(const uint8_t *, int len) { a += len; }
};
__device__ __forceinline__ int dec_len(long long v) {  // len(strconv.Itoa(v))
  const unsigned long long u = v < 0 ? 0ull - (unsigned long long)v : (unsigned long long)v;
  int d;
  if (u < 4294967296ull) {  // positions, counts: ten compares against immediates, no table in memory
    const uint32_t x = (uint32_t)u;
    d = 1 + (x >= 10u) + (x >= 100u) + (x >= 1000u) + (x >= 10000u) + (x >= 100000u) + (x >= 1000000u) + (x >= 10000000u) +
        (x >= 100000000u) + (x >= 1000000000u);
  } else {
    d = 10;
#pragma unroll 1
    while (d < 20 && u >= BVCF_P10[d]) d++;
  }
  return d + (v < 0 ? 1 : 0);
}
__device__ __forceinline__ void w_dec(CountWriter &w, long long v) { w.a += (uint32_t)dec_len(v); }

// ---- the text of a row that every cohort shares -----------------------------------------------------------
// "chrom \t pos \t type \t ref \t alt \t trTv \t" (main.go:570-606)
template <class W>
__device__ __forceinline__ void row_text_head(W &w, const LineCtx &lc, const OutAllele &oa) {
  // chrom (main.go:570-574)
  if (lc.chrom_n < 4 || lc.chrom[0] != 'c') w.packed(0x726863ull, 3);  // "chr"
  w.span(lc.chrom, lc.chrom_n);
  w.byte('\t');
  if (oa.pos_verbatim) w.span(lc.pos, lc.pos_n); else w_dec(w, oa.pos_val);
  if (lc.site_type != T_MULTI) {  // "\tSNP\t": the three-letter types as one piece
    const uint8_t *tt = (const uint8_t *)TYPE_TXT[lc.site_type];
    w.packed(0x09ull | ((uint64_t)tt[0] << 8) | ((uint64_t)tt[1] << 16) | ((uint64_t)tt[2] << 24) | (0x09ull << 32), 5);
  } else {
    w.byte('\t');
    w.span_const((const uint8_t *)TYPE_TXT[lc.site_type], TYPE_LEN[lc.site_type]);
    w.byte('\t');
  }
  const uint8_t trtv = lc.multi ? '0' : (oa.kind == 0 ? trtv_char(oa.ref, oa.alt_c) : '0');  // main.go:602-606
  if (oa.kind == 0) {  // "R\tA\tt\t" as one piece
    w.packed((uint64_t)oa.ref | (0x09ull << 8) | ((uint64_t)oa.alt_c << 16) | (0x09ull << 24) | ((uint64_t)trtv << 32) | (0x09ull << 40), 6);
  } else {
    w.byte(oa.ref);
    w.byte('\t');
    if (oa.kind == 1) { w.byte('+'); w.span(oa.ins_p, oa.ins_n); }
    else w_dec(w, oa.del_n);
    w.byte('\t');
    w.byte(trtv);
    w.byte('\t');
  }
}
// the --keepPos / --keepId / --keepInfo columns and the end of the row (main.go:671-692); INFO: the ALT index here,
// the span itself only when the writer goes straight to the output (staged rows get it at copy-out)
template <class W, bool INFO_SPAN, bool SPEC = false>
__device__ __forceinline__ void row_text_keep(W &w, const DevCfg &cfg, const LineCtx &lc, const OutAllele &oa) {
  if (SPEC) { w.byte('\n'); return; }
  if (cfg.keep_pos) { w.byte('\t'); w.span(lc.pos, lc.pos_n); }
  if (cfg.keep_id) { w.byte('\t'); w.span(lc.id, lc.id_n); }
  if (cfg.keep_info) {
    w.byte('\t'); w_dec(w, oa.alt_idx); w.byte('\t');
    if constexpr (INFO_SPAN) { w.span(lc.info, lc.info_n); w.byte('\n'); }
  } else {
    w.byte('\n');
  }
}

// ---- one output row (main.go:555-695) -------------------------------------------------------------------
// W = StageWriter: pass A (compose into the arena, or size only once the record has failed over to the slow path);
// W = GlobalWriter: pass C of a slow-path record.
template <class W, bool SPEC = false>
__device__ __forceinline__ void tile_emit_row(const TileParams &p, const LineRec &rec, const LineCtx &lc, const OutAllele &oa,
                                              GtStats &gs, int &gs_idx, W &w, RecOut &ro, const TileShared &sh, SlowOut &so) {
  const DevCfg &cfg = p.cfg;
  const bool want_tsv = SPEC ? true : (bool)cfg.want_tsv, keep_pos = SPEC ? false : (bool)cfg.keep_pos,
             keep_id = SPEC ? false : (bool)cfg.keep_id, keep_info = SPEC ? false : (bool)cfg.keep_info;
  const uint32_t fixed_w = SPEC ? 7u : (uint32_t)(cfg.name_fixed_w > 0 ? cfg.name_fixed_w : 0);  // name bytes, without the delimiter
  const uint32_t a = (uint32_t)oa.alt_idx + 1;
  const bool has_samples = cfg.n_samples > 0;
  if (has_samples) {
    if (gs_idx != oa.alt_idx) {  // MNP bases share their ALT index: reduce once (main.go:865-868)
      if (fixed_w > 0 && !(rec.flags & 1)) {
        // the scan kernel's inline summary is complete: only ALT #1 occurs among the samples
        gs.n_het = a == 1 ? rec.n_het1 : 0; gs.n_hom = a == 1 ? rec.n_hom1 : 0; gs.ac = a == 1 ? rec.ac1 : 0;
        gs.n_miss = rec.n_miss; gs.an = rec.an;
        gs.het_bytes = gs.n_het * fixed_w; gs.hom_bytes = gs.n_hom * fixed_w;
        gs.miss_bytes = gs.n_miss * fixed_w;
      } else if (a <= (uint32_t)STAT_ALLELES) {
        const LineStats &ls = p.stats[lc.li];
        gs.n_het = ls.n_het[a - 1]; gs.n_hom = ls.n_hom[a - 1]; gs.ac = ls.ac[a - 1];
        gs.het_bytes = ls.het_bytes[a - 1]; gs.hom_bytes = ls.hom_bytes[a - 1];
        gs.n_miss = ls.n_miss; gs.an = ls.an; gs.miss_bytes = ls.miss_bytes;
      } else {
        gs = reduce_events_thread(cfg, rec, p.events + rec.ev_start, lc.L, lc.content_len, a);
      }
      gs_idx = oa.alt_idx;
    }
    if (gs.ac == 0) return;  // main.go:558
  }
  const uint32_t dl = SPEC ? 1u : (uint32_t)cfg.delim_len;
  const uint32_t cnts[3] = {has_samples ? gs.n_het : 0u, has_samples ? gs.n_hom : 0u, has_samples ? gs.n_miss : 0u};
  const uint32_t nb[3] = {gs.het_bytes, gs.hom_bytes, gs.miss_bytes};
  uint32_t lb[3];  // list bytes
#pragma unroll
  for (int k = 0; k < 3; k++) lb[k] = (want_tsv && cnts[k]) ? nb[k] + (cnts[k] - 1) * dl : 0u;
  const bool big = has_samples && rec.ev_count > SMALL_EVENTS;  // lists and dosages are left to the names kernels
  const bool want_locus = SPEC ? false : (cfg.want_dosage && has_samples);
  const uint32_t tail = (want_tsv && keep_info) ? (uint32_t)lc.info_n + 1u : 0u;  // INFO span + EOL, never staged

  // ---- where the bytes go ----
  TRow *row = nullptr;
  uint32_t ri = ROW_NONE, a0 = 0;
  bool inline_lists = false;
  if constexpr (W::kStage) {
    if (!ro.failed) {
      // upper bound of the staged bytes: the constant pieces come to 100 bytes at most (3 "chr", 14 "\tMULTIALLELIC\t",
      // 6 ref/alt/trTv framing, 3 x 10 ratio columns, 30 ac/an/sampleMaf, 14 keepInfo framing, tabs, EOL)
      const uint32_t pos_b = oa.pos_verbatim ? (uint32_t)lc.pos_n : 20u;
      const uint32_t alt_b = oa.kind == 1 ? (uint32_t)oa.ins_n + 1u : 21u;
      uint32_t need = 0;
      if (want_tsv) {
        need = 104u + (uint32_t)lc.chrom_n + pos_b + alt_b + (has_samples ? 3u * (uint32_t)cfg.empty_len : (uint32_t)cfg.tail0_len) +
               (keep_pos ? (uint32_t)lc.pos_n : 0u) + (keep_id ? (uint32_t)lc.id_n : 0u);
        if (!big) need += lb[0] + lb[1] + lb[2];
      }
      if (want_locus) need += 8u + (uint32_t)lc.chrom_n + pos_b + alt_b;
      if (big) need += 16u;  // three counts, 4-byte aligned
      ri = ro.first == ROW_NONE ? (threadIdx.x & 31u) : atomicAdd(sh.rows_cur, 1u);
      const uint32_t off = atomicAdd(sh.arena_cur, (need + 15u) & ~15u);
      if (ri >= sh.rows_cap || off + need > sh.arena_cap) {
        ro.failed = true; ro.first = ROW_NONE;  // the whole record takes the slow path; keep sizing
      } else {
        row = &sh.rows[ri];
        a0 = sh.arena_s + off;
        inline_lists = !big && want_tsv;
      }
    }
    w.stg = row != nullptr;
    w.a = a0;
  }
  uint8_t *g_row0 = nullptr;
  if constexpr (!W::kStage) g_row0 = w.g;
  unsigned long long hole_total = 0;
  uint32_t la[3] = {0, 0, 0};                 // staged list starts (inline lists)
  uint32_t hpos[3] = {0, 0, 0}, hlen[3] = {0, 0, 0};
  unsigned long long dsts[3] = {~0ull, ~0ull, ~0ull};

  if (want_tsv) {
    row_text_head(w, lc, oa);
    if (!has_samples) {  // main.go:612-616,634-637,648-651,667: "! 0 ! 0 ! 0 0 0 0"
      w.span_const(cfg.tail0, cfg.tail0_len);  // composed once by the host
    } else {
      const uint32_t eff = (uint32_t)cfg.n_samples - gs.n_miss;  // main.go:563
      const uint32_t den[3] = {eff, eff, (uint32_t)cfg.n_samples};
#pragma unroll
      for (int k = 0; k < 3; k++) {
        if (cnts[k] == 0) {
          w.span_const(cfg.empty, cfg.empty_len); w.byte('\t'); w.byte('0');
        } else {
          if constexpr (W::kStage) {
            if (inline_lists) { la[k] = w.a; w.a += lb[k]; }      // filled below
            else { hpos[k] = w.a - a0; hlen[k] = lb[k]; hole_total += lb[k]; }
          } else {
            dsts[k] = (unsigned long long)(w.g - p.out);
            w.g += lb[k];                                          // filled by the names kernels
          }
          w.byte('\t');
          int fl;
          const uint64_t ft = format_ratio_g3(cnts[k], den[k], fl);
          w.packed(ft, fl);
        }
        w.byte('\t');
      }
      w_dec_small(w, gs.ac); w.byte('\t');
      w_dec_small(w, gs.an); w.byte('\t');
      if (gs.ac == 0) w.byte('0');
      else { int fl; const uint64_t ft = format_ratio_g3(gs.ac, gs.an, fl); w.packed(ft, fl); }
    }
    row_text_keep<W, !W::kStage, SPEC>(w, cfg, lc, oa);
  }

  uint32_t slen = 0, loc_len = 0;
  if constexpr (W::kStage) slen = w.a - a0;
  // ---- locus "chrom:pos:ref:alt" (main.go:577) ----
  if (want_locus) {
    if constexpr (W::kStage) {
      if (lc.chrom_n < 4 || lc.chrom[0] != 'c') w.packed(0x726863ull, 3);
      w.span(lc.chrom, lc.chrom_n);
      w.byte(':');
      if (oa.pos_verbatim) w.span(lc.pos, lc.pos_n); else w_dec(w, oa.pos_val);
      w.byte(':'); w.byte(oa.ref); w.byte(':');
      if (oa.kind == 0) w.byte(oa.alt_c);
      else if (oa.kind == 1) { w.byte('+'); w.span(oa.ins_p, oa.ins_n); }
      else w_dec(w, oa.del_n);
      loc_len = w.a - a0 - slen;
    } else {
      const unsigned long long gr = p.ctr->chunk_row_base + so.row;
      GlobalWriter lw;
      lw.g = p.loci + so.loci_off;
      lw.on = w.on && gr < p.dosage_cap_rows;
      uint8_t *const l0 = lw.g;
      // bytes beyond the locus buffer are counted, not written (the host grows the buffer and re-runs the chunk)
      unsigned long long room = so.loci_off < p.loci_cap ? p.loci_cap - so.loci_off : 0ull;
      const uint32_t worst = 8u + (uint32_t)lc.chrom_n + (oa.pos_verbatim ? (uint32_t)lc.pos_n : 20u) + (oa.kind == 1 ? (uint32_t)oa.ins_n + 1u : 21u);
      if (room < worst) lw.on = false;
      if (lc.chrom_n < 4 || lc.chrom[0] != 'c') lw.packed(0x726863ull, 3);
      lw.span(lc.chrom, lc.chrom_n);
      lw.byte(':');
      if (oa.pos_verbatim) lw.span(lc.pos, lc.pos_n); else w_dec(lw, oa.pos_val);
      lw.byte(':'); lw.byte(oa.ref); lw.byte(':');
      if (oa.kind == 0) lw.byte(oa.alt_c);
      else if (oa.kind == 1) { lw.byte('+'); lw.span(oa.ins_p, oa.ins_n); }
      else w_dec(lw, oa.del_n);
      loc_len = (uint32_t)(lw.g - l0);
      if (w.on && gr < p.dosage_cap_rows) p.loci_off[gr] = so.loci_off;
      so.loci_off += loc_len;
    }
  }

  // ---- row bookkeeping ----
  if constexpr (W::kStage) {
    ro.bytes += (unsigned long long)slen + hole_total + tail;
    ro.rows++;
    ro.loci += loc_len;
    if (big) ro.n_desc++;
    if (row) {
      row->hole_len[0] = hlen[0]; row->hole_len[1] = hlen[1]; row->hole_len[2] = hlen[2];
      if (big) {  // the names per list travel behind the staged bytes (RowDesc needs them at copy-out)
        const uint32_t ca = (w.a + 3u) & ~3u;
        sts32(ca, cnts[0]); sts32(ca + 4, cnts[1]); sts32(ca + 8, cnts[2]);
      }
      row->hole_pos[0] = (uint16_t)hpos[0]; row->hole_pos[1] = (uint16_t)hpos[1]; row->hole_pos[2] = (uint16_t)hpos[2];
      row->soff = (uint16_t)(a0 - sh.arena_s); row->slen = (uint16_t)slen; row->loc_len = (uint16_t)loc_len;
      row->next = (uint16_t)ROW_NONE; row->allele = (uint16_t)a;
      row->flags = (uint16_t)((tail ? 1u : 0u) | (big ? 2u : 0u));
      if (ro.first == ROW_NONE) ro.first = ri; else sh.rows[ro.last].next = (uint16_t)ri;
      ro.last = ri;
      if (inline_lists && (cnts[0] | cnts[1] | cnts[2])) fill_small_lists<SPEC>(p, rec, lc, a, la[0], la[1], la[2]);
    }
  } else {
    if (has_samples) {  // every row of a slow-path record is queued for the names kernels
      if (so.desc_ok) {
        RowDesc rd;
        rd.line = lc.li; rd.allele = a;
        rd.het_dst = dsts[0]; rd.hom_dst = dsts[1]; rd.miss_dst = dsts[2];
        rd.n_het = cnts[0]; rd.n_hom = cnts[1]; rd.n_miss = cnts[2];
        rd.row = (uint32_t)so.row;
        queue_row_desc(p, so.cls, so.desc, rd);
      }
      so.desc++;
    }
    so.row++;
    (void)g_row0;
  }
}

// ---- one record: field index, linePasses (main.go:447-454), the start of getAlleles ---------------------------
// Leaves the generator ready for gen_next (or done: filtered out / nothing to emit).
template <bool CACHE = true>
__device__ __forceinline__ void record_open(const TileParams &p, uint32_t li, const LineRec &rec, const uint8_t *s_filt,
                                            const uint32_t *s_filt_off, bool diag, LineCtx &lc, AlleleGen &g, DiagSink &ds,
                                            unsigned long long &line_no, uint32_t t[9]) {
  const DevCfg &cfg = p.cfg;
  const int n_filt = cfg.n_allow + cfg.n_excl;
  const uint8_t *L = p.in + rec.start;
  const uint32_t n = rec.len >= (uint32_t)cfg.eol_width ? rec.len - (uint32_t)cfg.eol_width : 0;  // main.go:535
  // ---- first eight/nine tabs (strings.Split, main.go:535) ----
  const int need = cfg.H - 1 < 9 ? cfg.H - 1 : 9;
  int found = need;
  bool far = false;  // a tab beyond 64 KiB from the line start: the scan kernel could not record it
#pragma unroll
  for (int k = 0; k < 9; k++) {
    t[k] = rec.tab[k];
    far = far || (k < need && t[k] == 0xFFFFu);
  }
  if (far) {
    found = 0;
    for (uint32_t i = 0; i < n && found < need; i++)
      if (L[i] == '\t') {
#pragma unroll
        for (int k = 0; k < 9; k++) if (k == found) t[k] = i;  // static indexing keeps t[] in registers
        found++;
      }
  }
  bool pass = found >= need;  // always true for scan-kernel records; defensive
#pragma unroll
  for (int k = 0; k < 9; k++) if (k >= found) t[k] = n;
  lc.L = L; lc.content_len = n; lc.li = li;
  lc.chrom = L; lc.chrom_n = (int)t[0];
  lc.pos = L + t[0] + 1; lc.pos_n = (int)(t[1] - t[0] - 1);
  lc.id = L + t[1] + 1; lc.id_n = (int)(t[2] - t[1] - 1);
  const uint8_t *ref = L + t[2] + 1; const int ref_n = (int)(t[3] - t[2] - 1);
  const uint8_t *alt = L + t[3] + 1; const int alt_n = (int)(t[4] - t[3] - 1);
  const uint8_t *filt = L + t[5] + 1; const int filt_n = (int)(t[6] - t[5] - 1);
  lc.info = L + t[6] + 1; lc.info_n = (int)(t[7] - t[6] - 1);
  lc.multi = false; lc.site_type = T_SNP;

  // ---- linePasses (main.go:447-454): exact whole-field match against the shared-memory table ----
  if (pass && (!cfg.allow_all || cfg.n_excl > 0)) {
    bool in_allow = false, in_excl = false;
    const bool fshort = filt_n <= 8;  // "PASS", ".", "q10": the field in a register, one round trip to memory
    const unsigned long long fw = (fshort && filt_n > 0) ? ld64_any(filt) : 0ull;
    for (int k = 0; k < n_filt; k++) {
      const uint32_t o = s_filt_off[k], ln = s_filt_off[k + 1] - o;
      bool eq = (int)ln == filt_n;
#pragma unroll 1
      for (int i = 0; eq && i < filt_n; i++) eq = s_filt[o + i] == (fshort ? (uint8_t)(fw >> (8 * i)) : filt[i]);
      if (eq) { if (k < cfg.n_allow) in_allow = true; else in_excl = true; }
    }
    if (!cfg.allow_all && !in_allow) pass = false;
    if (in_excl) pass = false;
  }

  // ---- getAlleles (main.go:723-1038) as a resumable generator ----
  g.ref = ref; g.alt = alt; g.ref_n = ref_n; g.alt_n = alt_n;
  g.s = 0; g.alt_idx = 0; g.mnp_i = -1; g.ta_off = 0; g.tn = 0; g.last = false;
  g.done = !(pass && ref_n > 0 && alt_n > 0);
  g.ipos = 0;
  // strconv.Atoi(POS) is only ever consulted when REF is longer than one base (main.go:752,822): SNPs and plain
  // insertions copy the POS text verbatim
  g.pos_ok = (g.done || ref_n <= 1) ? false : atoi_go(lc.pos, lc.pos_n, g.ipos);
  line_no = p.ctr->chunk_line_base + rec.ord;
  ds = p.diag;
  ds.line_start = rec.start;
  if (!g.done) gen_begin<CACHE>(g, lc, ds, line_no, diag);
  else g.cached = false;
}

// ---- one record, one thread: one converged tile_emit_row call site per output allele -------------------------
template <class W, bool SPEC = false>
__device__ __forceinline__ void tile_record(const TileParams &p, uint32_t li, const LineRec &rec, W &w, RecOut &ro,
                                            const TileShared &sh, SlowOut &so, const uint8_t *s_filt, const uint32_t *s_filt_off,
                                            bool diag, const uint8_t *&info_p, uint32_t &info_n) {
  LineCtx lc;
  AlleleGen g;
  DiagSink ds;
  unsigned long long line_no;
  uint32_t t[9];
  record_open(p, li, rec, s_filt, s_filt_off, diag, lc, g, ds, line_no, t);
  info_p = lc.info; info_n = (uint32_t)lc.info_n;
  GtStats gs;
  gs.n_het = gs.n_hom = gs.n_miss = gs.ac = gs.an = gs.het_bytes = gs.hom_bytes = gs.miss_bytes = 0;
  int gs_idx = -1;
  OutAllele oa;
  oa.ins_p = nullptr; oa.ins_n = 0; oa.del_n = 0; oa.pos_val = 0;
  while (gen_next(g, oa, ds, line_no, diag)) tile_emit_row<W, SPEC>(p, rec, lc, oa, gs, gs_idx, w, ro, sh, so);
}

// inclusive scan of v over the warp; the total in `total`
__device__ __forceinline__ unsigned long long warp_scan64(unsigned long long v, unsigned long long &total, int lane) {
  unsigned long long x = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const unsigned long long t = __shfl_up_sync(FULL, x, d);
    if (lane >= d) x += t;
  }
  total = __shfl_sync(FULL, x, 31);
  return x;
}

// shared memory per warp: arena (+ padding) and row table
__host__ __device__ constexpr uint32_t tile_smem_warp(uint32_t arena, uint32_t rows) { return arena + 16 + rows * (uint32_t)sizeof(TRow); }
constexpr uint32_t TILE_BLOCK_HDR = 32u * (uint32_t)sizeof(LaneRec);

// ---- compose ------------------------------------------------------------------------------------------------
// MINB resident CTAs per SM (sets the register budget), ARENA staging bytes and ROWS row descriptors per warp.
// Records with samples give about one row each (wide text: 10 KiB, 48 rows); sites-only input has a composer of its own
// (bvcf_compose_sites_kernel below).
template <int MINB, uint32_t ARENA, uint32_t ROWS, bool SPEC = false>
__global__ void __launch_bounds__(TILE_WARPS * 32, MINB) bvcf_compose_kernel(const __grid_constant__ TileParams p) {
  constexpr uint32_t TILE_ARENA = ARENA, TILE_ROWS = ROWS, TILE_SMEM_WARP = tile_smem_warp(ARENA, ROWS);
  static_assert(ROWS <= TILE_ROWS_MAX && ROWS >= TILE_THREADS, "row table size");
  extern __shared__ __align__(16) uint8_t s_dyn[];
  __shared__ uint8_t s_filt[FILT_SMEM];
  __shared__ uint32_t s_filt_off[65];
  __shared__ uint32_t s_cur[TILE_WARPS][2];   // per warp: arena bytes in use, next free row descriptor
  const DevCfg &cfg = p.cfg;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // FILTER allow/exclude table -> shared memory
  const int n_filt = cfg.n_allow + cfg.n_excl;
  for (int i = threadIdx.x; i < cfg.filt_bytes && i < FILT_SMEM; i += blockDim.x) s_filt[i] = cfg.filt_blob[i];
  for (int i = threadIdx.x; i <= n_filt && i < 65; i += blockDim.x) s_filt_off[i] = cfg.filt_off[i];
  __syncthreads();  // the only CTA barrier: from here on every warp is on its own
  if (p.ctr->ev_overflow | p.ctr->slot_overflow) return;  // the host grows the scratch and re-runs the chunk
  const uint32_t n_rec = p.ctr->chunk_records;
  const uint32_t n_tiles = (n_rec + TILE_THREADS - 1) / TILE_THREADS;
  const bool has_samples = cfg.n_samples > 0;
  uint8_t *const my_smem = s_dyn + (size_t)warp * TILE_SMEM_WARP;
  TRow *const s_rows = reinterpret_cast<TRow *>(my_smem + TILE_ARENA + 16);
  TileShared sh;
  sh.arena_s = (uint32_t)__cvta_generic_to_shared(my_smem);
  sh.arena_cap = TILE_ARENA;
  sh.rows_cap = TILE_ROWS;
  sh.rows = s_rows;
  sh.arena_cur = &s_cur[warp][0];
  sh.rows_cur = &s_cur[warp][1];

  // Tiles are handed out by a ticket counter (rows differ a lot in cost), two tickets ahead: a warp holds the next two
  // tiles it will compose.  The order was made for an L2 prefetch of those tiles' lines and events, which was measured
  // and dropped (no gain: the waits are dependent L1/L2 hits, not DRAM); it stays because the tile schedule is part of
  // every time measured on this kernel since, and taking one ticket per tile changes it.
  auto ticket = [&]() {
    uint32_t t = 0;
    if (lane == 0) t = atomicAdd(&p.ctr->tile_ticket, 1u);
    return __shfl_sync(FULL, t, 0);
  };
  uint32_t tile = ticket(), tile_n1 = ticket(), tile_n2;
  for (; tile < n_tiles; tile = tile_n1, tile_n1 = tile_n2) {
    if (lane == 0) { s_cur[warp][0] = 0; s_cur[warp][1] = TILE_THREADS; }
    tile_n2 = ticket();  // also orders the cursor reset before the lanes' allocations
    const uint32_t li = tile * TILE_THREADS + lane;
    const bool valid = li < n_rec;

    RecOut ro;
    ro.bytes = 0; ro.rows = 0; ro.loci = 0; ro.n_desc = 0; ro.first = ROW_NONE; ro.last = ROW_NONE; ro.failed = false;
    SlowOut so;
    so.row = 0; so.loci_off = 0; so.desc = 0; so.cls = 1; so.desc_ok = false;
    const uint8_t *info_p = nullptr;
    uint32_t info_n = 0, info_off = 0, ev_count = 0;
    if (valid) {
      const LineRec rec = p.lines[li];
      ev_count = rec.ev_count;
      StageWriter w;
      w.a = 0; w.stg = false;
      tile_record<StageWriter, SPEC>(p, li, rec, w, ro, sh, so, s_filt, s_filt_off, true, info_p, info_n);
      info_off = (uint32_t)(info_p - (p.in + rec.start));
    }
    const int cls = row_class(p, ev_count);
    if (ro.failed && has_samples) ro.n_desc = ro.rows;
    __syncwarp();  // every lane's staged bytes and row descriptors are in shared memory

    // ---- the tile's totals and its scratch block: 32 LaneRec | n_trows TRow | arena_used bytes ----
    const unsigned long long tot_b = warp_sum64(ro.bytes);
    const uint32_t tot_rows = __reduce_add_sync(FULL, ro.rows), tot_loci = __reduce_add_sync(FULL, ro.loci);
    const uint32_t tot_mid = __reduce_add_sync(FULL, cls == 0 ? ro.n_desc : 0u), tot_big = __reduce_add_sync(FULL, cls == 1 ? ro.n_desc : 0u),
                   tot_long = __reduce_add_sync(FULL, cls == 2 ? ro.n_desc : 0u);
    uint32_t arena_used = s_cur[warp][0], n_trows = s_cur[warp][1];
    if (arena_used > TILE_ARENA) arena_used = TILE_ARENA;   // failed allocations moved the cursor past the end
    if (n_trows > TILE_ROWS) n_trows = TILE_ROWS;
    arena_used = (arena_used + 15u) & ~15u;
    const uint32_t block_bytes = TILE_BLOCK_HDR + n_trows * (uint32_t)sizeof(TRow) + arena_used;
    unsigned long long soff = 0;
    if (lane == 0) soff = atomicAdd(reinterpret_cast<unsigned long long *>(&p.ctr->scratch_cursor), (unsigned long long)block_bytes);
    soff = __shfl_sync(FULL, soff, 0);
    const bool fits = soff + block_bytes <= p.scratch_cap;  // else: the host grows the scratch buffer and re-runs the chunk
    if (lane == 0) {
      TileAgg ag;
      ag.bytes = tot_b; ag.scratch_off = soff; ag.rows = tot_rows; ag.loci = tot_loci; ag.n_big = tot_big; ag.n_long = tot_long;
      ag.arena_used = arena_used; ag.n_trows = n_trows; ag.n_mid = tot_mid; ag.flags = 0;
      p.tile_agg[tile] = ag;
      if (!fits) p.ctr->scratch_overflow = 1;
    }
    if (fits) {
      uint8_t *blk = p.scratch + soff;
      LaneRec lr;
      lr.bytes = ro.bytes; lr.rows = ro.rows; lr.loci = ro.loci; lr.n_desc = ro.n_desc;
      lr.first = (uint16_t)ro.first; lr.flags = (uint16_t)((ro.failed ? 1u : 0u) | ((uint32_t)cls << 1));
      lr.info_off = info_off; lr.info_n = info_n;
      reinterpret_cast<LaneRec *>(blk)[lane] = lr;
      uint4 *dst = reinterpret_cast<uint4 *>(blk + TILE_BLOCK_HDR);
      const uint4 *rsrc = reinterpret_cast<const uint4 *>(s_rows);
      const uint32_t nrv = n_trows * (uint32_t)(sizeof(TRow) / 16);
      for (uint32_t i = lane; i < nrv; i += 32) dst[i] = rsrc[i];
      dst += nrv;
      const uint4 *asrc = reinterpret_cast<const uint4 *>(my_smem);
      const uint32_t nav = arena_used >> 4;
      for (uint32_t i = lane; i < nav; i += 32) dst[i] = asrc[i];
    }
    __syncwarp();  // every lane is done with the arena before the next tile's cursor reset
  }
}

// ---- compose, sites-only input ---------------------------------------------------------------------------------
// No samples: a row is its fixed columns, and 30 % of BASELINE's lines give two to eight of them.  With a thread per
// record a tile ran as long as its widest record (6.8 of 32 lanes active, 10,000 warp instructions per tile).  Here
// the generator still runs per record (phase B) but only PLANS the rows -- a 32-byte PendRow each, with the length of
// its text -- and the text is composed by whichever lane is free (phase C, a row per lane).  Because every length is
// known before a byte is written the rows land in the arena in output order, back to back: the tile's block is its
// output, and the copy-out kernel moves it with one coalesced warp copy (TileAgg::flags bit 0) -- unless --keepInfo
// interleaves INFO spans or a record overflowed to the slow path, which fall back to the row table.
struct __align__(16) PendRow {
  long long pos_val;
  uint32_t ins_off;       // kind 1: the inserted bases, offset from the line start
  int32_t n;              // kind 1: how many; kind 2: the (negative) deletion count
  uint32_t rel_off;       // text bytes of the record's rows before this one
  uint16_t len;           // text bytes of this row
  uint16_t next;          // next row of the record
  uint16_t alt_idx;
  uint8_t kind;           // OutAllele::kind, 0xFF: empty slot
  uint8_t ref, alt_c, verbatim, owner, pad;
};
static_assert(sizeof(PendRow) == sizeof(TRow), "a PendRow becomes a TRow in place");

template <class W>
__device__ __forceinline__ void sites_row_text(W &w, const DevCfg &cfg, const LineCtx &lc, const OutAllele &oa) {
  row_text_head(w, lc, oa);
  w.span_const(cfg.tail0, cfg.tail0_len);  // main.go:612-616,634-637,648-651,667: "! 0 ! 0 ! 0 0 0 0", composed once by the host
  row_text_keep<W, false>(w, cfg, lc, oa);
}

template <int MINB, uint32_t ARENA, uint32_t ROWS>
__global__ void __launch_bounds__(TILE_WARPS * 32, MINB) bvcf_compose_sites_kernel(const __grid_constant__ TileParams p) {
  constexpr uint32_t TILE_SMEM_WARP = tile_smem_warp(ARENA, ROWS);
  static_assert(ROWS <= TILE_ROWS_MAX && ROWS >= TILE_THREADS && ARENA < 65536u, "row table / arena size");
  extern __shared__ __align__(16) uint8_t s_dyn[];
  __shared__ uint8_t s_filt[FILT_SMEM];
  __shared__ uint32_t s_filt_off[65];
  __shared__ uint32_t s_next[TILE_WARPS];   // per warp: next free row slot
  const DevCfg &cfg = p.cfg;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int n_filt = cfg.n_allow + cfg.n_excl;
  for (int i = threadIdx.x; i < cfg.filt_bytes && i < FILT_SMEM; i += blockDim.x) s_filt[i] = cfg.filt_blob[i];
  for (int i = threadIdx.x; i <= n_filt && i < 65; i += blockDim.x) s_filt_off[i] = cfg.filt_off[i];
  __syncthreads();
  if (p.ctr->ev_overflow | p.ctr->slot_overflow) return;
  const uint32_t n_rec = p.ctr->chunk_records;
  const uint32_t n_tiles = (n_rec + TILE_THREADS - 1) / TILE_THREADS;
  uint8_t *const my_smem = s_dyn + (size_t)warp * TILE_SMEM_WARP;
  TRow *const s_rows = reinterpret_cast<TRow *>(my_smem + ARENA + 16);
  PendRow *const s_pend = reinterpret_cast<PendRow *>(s_rows);
  const uint32_t arena_s = (uint32_t)__cvta_generic_to_shared(my_smem);
  const uint32_t tail = (cfg.want_tsv && cfg.keep_info) ? 1u : 0u;  // INFO span + EOL appended at copy-out

  for (;;) {
    uint32_t tile = 0;
    if (lane == 0) { tile = atomicAdd(&p.ctr->tile_ticket, 1u); s_next[warp] = TILE_THREADS; }
    tile = __shfl_sync(FULL, tile, 0);
    __syncwarp();  // the cursor reset before the lanes' allocations
    if (tile >= n_tiles) break;
    const uint32_t li = tile * TILE_THREADS + lane;
    const bool valid = li < n_rec;

    // ---- phase B: a record per lane plans its rows ----
    s_pend[lane].kind = 0xFF;
    uint32_t n_rows = 0, last = ROW_NONE, first = ROW_NONE, info_n = 0, info_off = 0;
    unsigned long long staged = 0, start = 0;
    uint32_t t0 = 0, t1 = 0, t2 = 0, misc = 0;
    bool failed = false;
    if (valid) {
      const LineRec rec = p.lines[li];
      LineCtx lc;
      AlleleGen g;
      DiagSink ds;
      unsigned long long line_no;
      uint32_t t[9];
      record_open<false>(p, li, rec, s_filt, s_filt_off, true, lc, g, ds, line_no, t);  // REF / ALT in registers spill at 64
      start = rec.start; t0 = t[0]; t1 = t[1]; t2 = t[2];
      info_n = (uint32_t)lc.info_n; info_off = t[6] + 1;
      OutAllele oa;
      oa.ins_p = lc.L; oa.ins_n = 0; oa.del_n = 0; oa.pos_val = 0;
      while (gen_next(g, oa, ds, line_no, true)) {
        CountWriter cw;
        cw.a = 0;
        if (cfg.want_tsv) sites_row_text(cw, cfg, lc, oa);
        if (!failed) {
          const uint32_t slot = n_rows == 0 ? (uint32_t)lane : atomicAdd(&s_next[warp], 1u);
          if (slot >= ROWS) {
            failed = true;  // slow path; the sizes stay exact
          } else if (cw.a > 0xFFFFu || staged > 0xFFFFFFFFull || oa.alt_idx > 0xFFFF) {
            failed = true;
            s_pend[slot].kind = 0xFF;
          } else {
            PendRow pr;
            pr.pos_val = oa.pos_val;
            pr.ins_off = oa.kind == 1 ? (uint32_t)(oa.ins_p - lc.L) : 0u;
            pr.n = oa.kind == 1 ? (int32_t)oa.ins_n : (int32_t)oa.del_n;
            pr.rel_off = (uint32_t)staged; pr.len = (uint16_t)cw.a; pr.next = (uint16_t)ROW_NONE;
            pr.alt_idx = (uint16_t)oa.alt_idx; pr.kind = (uint8_t)oa.kind; pr.ref = oa.ref; pr.alt_c = oa.alt_c;
            pr.verbatim = oa.pos_verbatim ? 1 : 0; pr.owner = (uint8_t)lane; pr.pad = 0;
            s_pend[slot] = pr;
            if (n_rows) s_pend[last].next = (uint16_t)slot; else first = slot;
            last = slot;
          }
        }
        staged += cw.a;
        n_rows++;
      }
      misc = (uint32_t)lc.site_type | (lc.multi ? 0x100u : 0u);
    }
    __syncwarp();

    // ---- the arena in output order: records one after the other, a record's rows back to back ----
    failed = failed || staged > ARENA;
    const uint32_t mine = failed ? 0u : (uint32_t)staged;
    uint32_t incl = mine;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const uint32_t v = __shfl_up_sync(FULL, incl, d);
      if (lane >= d) incl += v;
    }
    if (!failed && incl > ARENA) failed = true;  // the tail of an overfull tile
    const uint32_t base = incl - mine;
    const uint32_t fmask = __ballot_sync(FULL, failed && n_rows > 0);
    uint32_t arena_used = __reduce_max_sync(FULL, failed ? 0u : incl);
    uint32_t n_slots = s_next[warp];
    if (n_slots > ROWS) n_slots = ROWS;
    const bool dense = fmask == 0u && tail == 0u;

    // ---- phase C: a row per lane composes its text ----
    for (uint32_t r0 = 0; r0 < n_slots; r0 += 32) {
      const uint32_t r = r0 + lane;
      PendRow pr;
      pr.kind = 0xFF; pr.owner = (uint8_t)lane;
      if (r < n_slots) pr = s_pend[r];
      const int owner = pr.kind == 0xFF ? lane : (int)pr.owner;
      const unsigned long long o_start = __shfl_sync(FULL, start, owner);
      const uint32_t o_t0 = __shfl_sync(FULL, t0, owner), o_t1 = __shfl_sync(FULL, t1, owner), o_t2 = __shfl_sync(FULL, t2, owner);
      const uint32_t o_misc = __shfl_sync(FULL, misc, owner), o_base = __shfl_sync(FULL, base, owner);
      if (pr.kind != 0xFF && !((fmask >> owner) & 1u)) {
        LineCtx lc;
        lc.L = p.in + o_start; lc.content_len = 0; lc.li = 0;
        lc.chrom = lc.L; lc.chrom_n = (int)o_t0;
        lc.pos = lc.L + o_t0 + 1; lc.pos_n = (int)(o_t1 - o_t0 - 1);
        lc.id = lc.L + o_t1 + 1; lc.id_n = (int)(o_t2 - o_t1 - 1);
        lc.info = lc.L; lc.info_n = 0;
        lc.site_type = (int)(o_misc & 0xFFu); lc.multi = (o_misc & 0x100u) != 0;
        OutAllele oa;
        oa.pos_val = pr.pos_val; oa.ins_p = lc.L + pr.ins_off; oa.ins_n = pr.kind == 1 ? pr.n : 0;
        oa.del_n = pr.kind == 2 ? (long long)pr.n : 0; oa.alt_idx = pr.alt_idx; oa.kind = pr.kind;
        oa.ref = pr.ref; oa.alt_c = pr.alt_c; oa.pos_verbatim = pr.verbatim != 0;
        StageWriter w;
        w.stg = true; w.a = arena_s + o_base + pr.rel_off;
        if (cfg.want_tsv) sites_row_text(w, cfg, lc, oa);
        if (!dense) {
          TRow tr;
          tr.hole_len[0] = tr.hole_len[1] = tr.hole_len[2] = 0;
          tr.hole_pos[0] = tr.hole_pos[1] = tr.hole_pos[2] = 0;
          tr.soff = (uint16_t)(o_base + pr.rel_off); tr.slen = pr.len; tr.loc_len = 0;
          tr.next = pr.next; tr.allele = (uint16_t)(pr.alt_idx + 1u); tr.flags = (uint16_t)tail; tr.pad = 0;
          s_rows[r] = tr;
        }
      }
    }
    __syncwarp();

    // ---- the tile's totals and its scratch block ----
    const unsigned long long bytes = staged + (tail ? (unsigned long long)n_rows * (info_n + 1ull) : 0ull);
    const unsigned long long tot_b = warp_sum64(bytes);
    const uint32_t tot_rows = __reduce_add_sync(FULL, n_rows);
    arena_used = (arena_used + 15u) & ~15u;
    const uint32_t n_trows = dense ? 0u : n_slots;
    const uint32_t block_bytes = dense ? arena_used : TILE_BLOCK_HDR + n_trows * (uint32_t)sizeof(TRow) + arena_used;
    unsigned long long soff = 0;
    if (lane == 0) soff = atomicAdd(reinterpret_cast<unsigned long long *>(&p.ctr->scratch_cursor), (unsigned long long)block_bytes);
    soff = __shfl_sync(FULL, soff, 0);
    const bool fits = soff + block_bytes <= p.scratch_cap;
    if (lane == 0) {
      TileAgg ag;
      ag.bytes = tot_b; ag.scratch_off = soff; ag.rows = tot_rows; ag.loci = 0; ag.n_big = 0; ag.n_long = 0;
      ag.arena_used = arena_used; ag.n_trows = n_trows; ag.n_mid = 0; ag.flags = dense ? 1u : 0u;
      p.tile_agg[tile] = ag;
      if (!fits) p.ctr->scratch_overflow = 1;
    }
    if (fits) {
      uint8_t *blk = p.scratch + soff;
      uint4 *dst = reinterpret_cast<uint4 *>(blk);
      if (!dense) {
        LaneRec lr;
        lr.bytes = bytes; lr.rows = n_rows; lr.loci = 0; lr.n_desc = 0;
        lr.first = (uint16_t)(failed ? ROW_NONE : first); lr.flags = (uint16_t)((failed ? 1u : 0u) | (1u << 1));
        lr.info_off = info_off; lr.info_n = info_n;
        reinterpret_cast<LaneRec *>(blk)[lane] = lr;
        dst = reinterpret_cast<uint4 *>(blk + TILE_BLOCK_HDR);
        const uint4 *rsrc = reinterpret_cast<const uint4 *>(s_rows);
        const uint32_t nrv = n_trows * (uint32_t)(sizeof(TRow) / 16);
        for (uint32_t i = lane; i < nrv; i += 32) dst[i] = rsrc[i];
        dst += nrv;
      }
      const uint4 *asrc = reinterpret_cast<const uint4 *>(my_smem);
      const uint32_t nav = arena_used >> 4;
      for (uint32_t i = lane; i < nav; i += 32) dst[i] = asrc[i];
    }
    __syncwarp();  // every lane is done with the arena and the row table before the next tile
  }
}

// ---- tile offsets: exclusive scan of the tile totals (five quantities) over the sub-chunk's tiles ------------
constexpr int TSCAN_BLOCKS = 148, TSCAN_THREADS = 256;
constexpr int TQ = 6;  // quantities scanned: bytes, locus bytes, rows, mid / big / long queued rows
__device__ __forceinline__ void tot_of(const TileAgg &a, unsigned long long v[TQ]) {
  v[0] = a.bytes; v[1] = a.loci; v[2] = a.rows; v[3] = a.n_big; v[4] = a.n_long; v[5] = a.n_mid;
}
__device__ __forceinline__ void tscan_span(uint32_t n_tiles, uint32_t &lo, uint32_t &hi) {
  const uint32_t span = (n_tiles + TSCAN_BLOCKS - 1) / TSCAN_BLOCKS;
  const unsigned long long l = (unsigned long long)blockIdx.x * span;
  lo = l > n_tiles ? n_tiles : (uint32_t)l;
  hi = l + span > n_tiles ? n_tiles : (uint32_t)(l + span);
}
__global__ void __launch_bounds__(TSCAN_THREADS) bvcf_tile_reduce_kernel(const __grid_constant__ TileParams p) {
  __shared__ unsigned long long s_w[TQ][TSCAN_THREADS / 32];
  if (p.ctr->ev_overflow | p.ctr->slot_overflow) return;
  const uint32_t n_tiles = (p.ctr->chunk_records + TILE_THREADS - 1) / TILE_THREADS;
  uint32_t lo, hi;
  tscan_span(n_tiles, lo, hi);
  unsigned long long s[TQ] = {0, 0, 0, 0, 0, 0};
  for (uint32_t t = lo + threadIdx.x; t < hi; t += TSCAN_THREADS) {
    unsigned long long v[TQ];
    tot_of(p.tile_agg[t], v);
#pragma unroll
    for (int k = 0; k < TQ; k++) s[k] += v[k];
  }
#pragma unroll
  for (int k = 0; k < TQ; k++) {
    const unsigned long long w = warp_sum64(s[k]);
    if ((threadIdx.x & 31) == 0) s_w[k][threadIdx.x >> 5] = w;
  }
  __syncthreads();
  if (threadIdx.x < TQ) {
    unsigned long long t = 0;
    for (int i = 0; i < TSCAN_THREADS / 32; i++) t += s_w[threadIdx.x][i];
    p.tile_partial[TQ * blockIdx.x + threadIdx.x] = t;
  }
}
// one warp: exclusive scan of the TSCAN_BLOCKS span totals; advances the run's cursors, raises the capacity flags
__global__ void __launch_bounds__(32) bvcf_tile_spine_kernel(const __grid_constant__ TileParams p) {
  RunCounters *c = p.ctr;
  if (c->ev_overflow | c->slot_overflow) return;
  const int lane = threadIdx.x;
  unsigned long long run[TQ] = {0, 0, 0, 0, 0, 0};
  for (int base = 0; base < TSCAN_BLOCKS; base += 32) {
    const int b = base + lane;
#pragma unroll
    for (int k = 0; k < TQ; k++) {
      const unsigned long long v = b < TSCAN_BLOCKS ? p.tile_partial[TQ * b + k] : 0ull;
      unsigned long long tot;
      const unsigned long long inc = warp_scan64(v, tot, lane);
      if (b < TSCAN_BLOCKS) p.tile_partial[TQ * b + k] = run[k] + inc - v;
      run[k] += tot;
    }
  }
  if (lane == 0) {
    c->out_cursor = c->chunk_out_base + run[0];
    c->loci_cursor = c->chunk_loci_base + run[1];
    c->row_cursor = c->chunk_row_base + run[2];
    c->n_big_rows = (unsigned int)run[3];
    c->n_long_rows = (unsigned int)run[4];
    c->n_mid_rows = (unsigned int)run[5];
    if (c->out_cursor > p.out_cap) c->out_overflow = 1;
    if (run[3] + run[4] + run[5] > p.row_desc_cap) c->row_overflow = 1;
  }
}
__global__ void __launch_bounds__(TSCAN_THREADS) bvcf_tile_offsets_kernel(const __grid_constant__ TileParams p) {
  __shared__ unsigned long long s_w[TQ][TSCAN_THREADS / 32];
  if (p.ctr->ev_overflow | p.ctr->slot_overflow) return;
  const uint32_t n_tiles = (p.ctr->chunk_records + TILE_THREADS - 1) / TILE_THREADS;
  uint32_t lo, hi;
  tscan_span(n_tiles, lo, hi);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned long long run[TQ];
#pragma unroll
  for (int k = 0; k < TQ; k++) run[k] = p.tile_partial[TQ * blockIdx.x + k];
  for (uint32_t base = lo; base < hi; base += TSCAN_THREADS) {
    const uint32_t t = base + threadIdx.x;
    unsigned long long in[TQ] = {0, 0, 0, 0, 0, 0};
    if (t < hi) tot_of(p.tile_agg[t], in);
    unsigned long long inc[TQ], wt[TQ];
#pragma unroll
    for (int k = 0; k < TQ; k++) inc[k] = warp_scan64(in[k], wt[k], lane);
    __syncthreads();
    if (lane == 0) {
#pragma unroll
      for (int k = 0; k < TQ; k++) s_w[k][warp] = wt[k];
    }
    __syncthreads();
    unsigned long long ex[TQ];
#pragma unroll
    for (int k = 0; k < TQ; k++) {
      unsigned long long off = 0, tot = 0;
#pragma unroll
      for (int i = 0; i < TSCAN_THREADS / 32; i++) {
        const unsigned long long wv = s_w[k][i];
        if (i < warp) off += wv;
        tot += wv;
      }
      ex[k] = run[k] + off + inc[k] - in[k];
      run[k] += tot;
    }
    if (t < hi) {
      TileBase b;
      b.bytes = ex[0]; b.loci = ex[1]; b.rows = (uint32_t)ex[2]; b.n_big = (uint32_t)ex[3]; b.n_long = (uint32_t)ex[4];
      b.n_mid = (uint32_t)ex[5];
      p.tile_base[t] = b;
    }
  }
}

// ---- dosage rows start as all-reference (main.go:576-584: a row of zeros, then the non-reference samples) ---------
// The sub-chunk's rows [chunk_row_base, row_cursor) x n_samples bytes, known once the tile spine has run: plain 16-byte
// stores at memory speed, 15.5 GB of them at C5.  (Zeroing each tile's rows inside the copy-out kernel, which runs at
// half occupancy and waits on its loads, was no slower in total: 6.09 against 5.93 ms for the two together.)
__global__ void __launch_bounds__(256) bvcf_dosage_zero_kernel(const __grid_constant__ TileParams p) {
  const RunCounters *c = p.ctr;
  if (c->ev_overflow | c->slot_overflow | c->out_overflow | c->row_overflow | c->scratch_overflow) return;
  if (!p.dosage || p.cfg.n_samples <= 0) return;
  unsigned long long r_lo = c->chunk_row_base, r_hi = c->row_cursor;
  if (r_hi > p.dosage_cap_rows) r_hi = p.dosage_cap_rows;
  if (r_lo >= r_hi) return;
  const unsigned long long ns = (unsigned long long)p.cfg.n_samples;
  uint8_t *const base = reinterpret_cast<uint8_t *>(p.dosage);
  const unsigned long long b0 = r_lo * ns, b1 = r_hi * ns;
  const unsigned long long a0 = (b0 + 15ull) & ~15ull, a1 = b1 & ~15ull;  // cudaMalloc'ed: base is 256-byte aligned
  const unsigned long long tid = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x, nth = (unsigned long long)gridDim.x * blockDim.x;
  if (a0 >= a1) {
    for (unsigned long long i = b0 + tid; i < b1; i += nth) base[i] = 0;
    return;
  }
  for (unsigned long long i = b0 + tid; i < a0; i += nth) base[i] = 0;
  uint4 *v = reinterpret_cast<uint4 *>(base + a0);
  const unsigned long long nv = (a1 - a0) >> 4;
  for (unsigned long long i = tid; i < nv; i += nth) v[i] = make_uint4(0u, 0u, 0u, 0u);
  for (unsigned long long i = a1 + tid; i < b1; i += nth) base[i] = 0;
}

// ---- copy-out -----------------------------------------------------------------------------------------------
// No shared memory and few registers: the staged bytes are read straight from the tile's scratch block (L2), so the
// kernel runs at full occupancy and hides those latencies with warps instead.
__device__ __forceinline__ TRow ld_trow(const uint8_t *p) {
  const uint4 a = reinterpret_cast<const uint4 *>(p)[0], b = reinterpret_cast<const uint4 *>(p)[1];
  TRow t;
  t.hole_len[0] = a.x; t.hole_len[1] = a.y; t.hole_len[2] = a.z;
  t.hole_pos[0] = (uint16_t)a.w; t.hole_pos[1] = (uint16_t)(a.w >> 16);
  t.hole_pos[2] = (uint16_t)b.x; t.soff = (uint16_t)(b.x >> 16);
  t.slen = (uint16_t)b.y; t.loc_len = (uint16_t)(b.y >> 16);
  t.next = (uint16_t)b.z; t.allele = (uint16_t)(b.z >> 16);
  t.flags = (uint16_t)b.w; t.pad = 0;
  return t;
}
// n bytes of a tile's scratch block (16-byte aligned, padded) to any address, the whole warp: aligned 16-byte stores
__device__ __forceinline__ void warp_copy_out(uint8_t *d, const uint8_t *s, uint32_t n, int lane) {
  uint32_t head = (uint32_t)((0u - (uintptr_t)d) & 15u);
  if (head > n) head = n;
  if ((uint32_t)lane < head) d[lane] = s[lane];
  d += head; s += head; n -= head;
  const uint32_t nv = n >> 4;
  const uint32_t sh = (uint32_t)((uintptr_t)s & 3u) * 8u;
  const uint32_t *wp = reinterpret_cast<const uint32_t *>((uintptr_t)s & ~(uintptr_t)3);
  uint4 *dv = reinterpret_cast<uint4 *>(d);
  for (uint32_t v = lane; v < nv; v += 32) {
    const uint32_t *q = wp + 4 * v;
    const uint32_t w0 = q[0], w1 = q[1], w2 = q[2], w3 = q[3], w4 = q[4];
    dv[v] = make_uint4(__funnelshift_r(w0, w1, sh), __funnelshift_r(w1, w2, sh), __funnelshift_r(w2, w3, sh), __funnelshift_r(w3, w4, sh));
  }
  const uint32_t done = nv << 4, rest = n - done;
  if ((uint32_t)lane < rest) d[done + lane] = s[done + lane];
}
__global__ void __launch_bounds__(TILE_WARPS * 32, 8) bvcf_copyout_kernel(const __grid_constant__ TileParams p) {
  const DevCfg &cfg = p.cfg;
  const int lane = threadIdx.x & 31;
  const RunCounters *c = p.ctr;
  // any capacity miss: the host grows the buffer and re-runs the chunk
  if (c->ev_overflow | c->slot_overflow | c->out_overflow | c->row_overflow | c->scratch_overflow) return;
  const uint32_t n_rec = c->chunk_records;
  const uint32_t n_tiles = (n_rec + TILE_THREADS - 1) / TILE_THREADS;
  const unsigned long long out_base = c->chunk_out_base, row0 = c->chunk_row_base, loci0 = c->chunk_loci_base;
  const bool has_samples = cfg.n_samples > 0;
  const bool want_locus = cfg.want_dosage && has_samples;

  // tiles by ticket, one ahead: the next tile's totals are loaded while this one is copied
  auto ticket = [&]() {
    uint32_t t = 0;
    if (lane == 0) t = atomicAdd(&p.ctr->tile_ticket2, 1u);
    return __shfl_sync(FULL, t, 0);
  };
  uint32_t tile = ticket(), tile_n1 = ticket();
  TileAgg ag_next;
  ag_next.bytes = 0; ag_next.scratch_off = 0; ag_next.rows = ag_next.loci = ag_next.n_big = ag_next.n_long = 0;
  ag_next.arena_used = ag_next.n_trows = 0; ag_next.n_mid = 0; ag_next.flags = 0;
  if (tile < n_tiles) ag_next = p.tile_agg[tile];
  for (; tile < n_tiles; tile = tile_n1, tile_n1 = ticket()) {
    const TileAgg ag = ag_next;
    const bool more = tile_n1 < n_tiles;
    if (more) ag_next = p.tile_agg[tile_n1];  // consumed further down, after this tile's own loads
    const TileBase tb = p.tile_base[tile];
    const uint8_t *blk = p.scratch + ag.scratch_off;
    if (ag.flags & 1u) {  // a dense block: the tile's output bytes, in order
      warp_copy_out(p.out + out_base + tb.bytes, blk, (uint32_t)ag.bytes, lane);
      continue;
    }
    const LaneRec lr = reinterpret_cast<const LaneRec *>(blk)[lane];
    const uint8_t *rows_g = blk + TILE_BLOCK_HDR;
    const uint8_t *arena_g = rows_g + (size_t)ag.n_trows * sizeof(TRow);
    const uint32_t li = tile * TILE_THREADS + lane;
    const bool failed = lr.flags & 1u;
    const int cls = (int)((lr.flags >> 1) & 3u);
    unsigned long long tot;
    const unsigned long long in_b = warp_scan64(lr.bytes, tot, lane);
    const unsigned long long in_rl = warp_scan64((unsigned long long)lr.rows | ((unsigned long long)lr.loci << 32), tot, lane);
    const unsigned long long in_d = warp_scan64(cls == 1 ? ((unsigned long long)lr.n_desc << 32) : (cls == 0 ? (unsigned long long)lr.n_desc : 0ull), tot, lane);
    const unsigned long long in_l = warp_scan64(cls == 2 ? (unsigned long long)lr.n_desc : 0ull, tot, lane);

    // (the tile's dosage rows were zeroed by bvcf_dosage_zero_kernel: all-reference; the small rows' samples are
    // scattered below, the queued rows' by the names kernels)
    if (li < n_rec && lr.rows) {
      unsigned long long off = out_base + tb.bytes + (in_b - lr.bytes);           // first output byte of this record
      unsigned long long r = (unsigned long long)tb.rows + ((uint32_t)in_rl - lr.rows);  // its first row within the sub-chunk
      unsigned long long lo = loci0 + tb.loci + ((uint32_t)(in_rl >> 32) - lr.loci);
      uint32_t d_ord = cls == 2 ? tb.n_long + ((uint32_t)in_l - lr.n_desc)
                                : (cls == 1 ? tb.n_big + ((uint32_t)(in_d >> 32) - lr.n_desc) : tb.n_mid + ((uint32_t)in_d - lr.n_desc));
      if (!failed) {
        const uint8_t *line = nullptr;
        for (uint32_t ri = lr.first; ri != ROW_NONE;) {
          const TRow t = ld_trow(rows_g + (size_t)ri * sizeof(TRow));
          const uint8_t *sa = arena_g + t.soff;
          unsigned long long dsts[3] = {~0ull, ~0ull, ~0ull};
          unsigned long long row_bytes = t.slen;
          {
            uint8_t *g = p.out + off;
            uint32_t pos = 0;
            if (t.hole_len[0] | t.hole_len[1] | t.hole_len[2]) {
#pragma unroll
              for (int k = 0; k < 3; k++) {
                if (t.hole_len[k]) {
                  copy_g2g(g, sa + pos, t.hole_pos[k] - pos);
                  g += t.hole_pos[k] - pos;
                  pos = t.hole_pos[k];
                  dsts[k] = (unsigned long long)(g - p.out);
                  g += t.hole_len[k];
                }
              }
            }
            copy_g2g(g, sa + pos, t.slen - pos);
            g += t.slen - pos;
            if (t.flags & 1u) {  // INFO straight from the input line, then the EOL (main.go:684-692)
              if (!line) line = p.in + p.lines[li].start;
              copy_g2g(g, line + lr.info_off, lr.info_n);
              g[lr.info_n] = '\n';
            }
          }
          row_bytes += (unsigned long long)t.hole_len[0] + t.hole_len[1] + t.hole_len[2] + ((t.flags & 1u) ? lr.info_n + 1u : 0u);
          const unsigned long long gr = row0 + r;
          if (want_locus && gr < p.dosage_cap_rows) {
            if (lo + t.loc_len <= p.loci_cap) copy_g2g(p.loci + lo, sa + t.slen, t.loc_len);
            p.loci_off[gr] = lo;
            if (!(t.flags & 2u) && p.dosage) small_dosage(p, p.lines[li], t.allele, p.dosage + gr * (unsigned long long)cfg.n_samples);
          }
          if (t.flags & 2u) {
            const uint32_t *cnt = reinterpret_cast<const uint32_t *>(arena_g + ((t.soff + t.slen + t.loc_len + 3u) & ~3u));
            RowDesc rd;
            rd.line = li; rd.allele = t.allele;
            rd.het_dst = dsts[0]; rd.hom_dst = dsts[1]; rd.miss_dst = dsts[2];
            rd.n_het = cnt[0]; rd.n_hom = cnt[1]; rd.n_miss = cnt[2];
            rd.row = (uint32_t)r;
            queue_row_desc(p, cls, d_ord, rd);
            d_ord++;
          }
          off += row_bytes; r++; lo += t.loc_len;
          ri = t.next;
        }
      } else {
        // slow path: the record is written by bvcf_slow_rows_kernel at these places
        const uint32_t k = atomicAdd(&p.ctr->n_slow, 1u);
        if (k < p.slow_cap) {
          SlowRec sr;
          sr.out_off = off; sr.loci_off = lo; sr.li = li; sr.row = (uint32_t)r; sr.desc = d_ord; sr.flags = 1u | ((uint32_t)cls << 1);
          p.slow[k] = sr;
        }
      }
    }
  }
}

// ---- slow path: one thread per record, bytes straight to global memory --------------------------------------
__global__ void __launch_bounds__(64) bvcf_slow_rows_kernel(const __grid_constant__ TileParams p) {
  __shared__ uint8_t s_filt[FILT_SMEM];
  __shared__ uint32_t s_filt_off[65];
  const DevCfg &cfg = p.cfg;
  const int n_filt = cfg.n_allow + cfg.n_excl;
  for (int i = threadIdx.x; i < cfg.filt_bytes && i < FILT_SMEM; i += blockDim.x) s_filt[i] = cfg.filt_blob[i];
  for (int i = threadIdx.x; i <= n_filt && i < 65; i += blockDim.x) s_filt_off[i] = cfg.filt_off[i];
  __syncthreads();
  const RunCounters *c = p.ctr;
  if (c->ev_overflow | c->slot_overflow | c->out_overflow | c->row_overflow | c->scratch_overflow) return;
  uint32_t n = c->n_slow;
  if (n > p.slow_cap) n = p.slow_cap;  // flagged below; the host re-runs the chunk with a larger list
  if (blockIdx.x == 0 && threadIdx.x == 0 && c->n_slow > p.slow_cap) p.ctr->slow_overflow = 1;
  TileShared sh;
  sh.arena_s = 0; sh.arena_cap = 0; sh.rows_cap = 0; sh.rows = nullptr; sh.arena_cur = nullptr; sh.rows_cur = nullptr;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const SlowRec sr = p.slow[i];
    const LineRec rec = p.lines[sr.li];
    GlobalWriter gw;
    gw.g = p.out + sr.out_off; gw.on = true;
    SlowOut so;
    so.row = sr.row; so.loci_off = sr.loci_off; so.desc = sr.desc; so.cls = (int)((sr.flags >> 1) & 3u); so.desc_ok = true;
    RecOut ro;
    ro.bytes = 0; ro.rows = 0; ro.loci = 0; ro.n_desc = 0; ro.first = ROW_NONE; ro.last = ROW_NONE; ro.failed = true;
    const uint8_t *info_p;
    uint32_t info_n;
    tile_record<GlobalWriter>(p, sr.li, rec, gw, ro, sh, so, s_filt, s_filt_off, false, info_p, info_n);
  }
}

}  // namespace bvcf
