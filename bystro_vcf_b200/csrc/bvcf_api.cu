// bvcf_api.cu -- host side of libbvcf: contexts, staging slots, the kernel pipeline and the C ABI.
//
// Pipeline per sub-chunk (all launches on one stream, no host synchronisation in between):
//   bvcf_scan_genotype_kernel      index + genotype events                    (north-star kernels 1+3)
//   bvcf_prefix_* (mode 0)         per-range record counts -> bases
//   bvcf_compact_lines_kernel      input-ordered line table
//   bvcf_line_stats_{,big_}kernel  genotype summaries the scan could not finish inline
//   bvcf_compose_kernel            FILTER + getAlleles + row text + short name lists, staged per tile of 32 records
//   bvcf_tile_{reduce,spine,offsets}  tile totals -> output offsets, cursors            (north-star kernels 2+4)
//   bvcf_dosage_zero_kernel        the sub-chunk's dosage rows start as zeros (only with --dosageOutput)
//   bvcf_copyout_kernel            rows to the output with aligned stores, loci, RowDesc work lists
//   bvcf_slow_rows_kernel          the few records that do not fit a tile's arena
//   bvcf_names_{vec,long,big}_     long sample-name lists, their dosage rows  (north-star kernel 4b)
// A bgzf chunk (bvcf_submit_bgzf) is inflated on the same stream first (bvcf_inflate_kernel, into the slot's input
// buffer); bvcf_diag_fields_kernel gathers the CHROM and POS fields of its diagnosed lines for the host's log lines.
#include "../../include/bvcf.h"

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "bvcf_common.cuh"
#include "bvcf_prefix.cuh"
#include "bvcf_rows.cuh"
#include "bvcf_tile.cuh"
#include "bvcf_names.cuh"
#include "bvcf_scan.cuh"
#include "bvcf_inflate.cuh"
#include "bvcf_deflate.cuh"

using namespace bvcf;

namespace {

struct DevBuf {
  void *p = nullptr;
  size_t cap = 0;
};

struct Scratch {
  // geometry
  uint64_t sub_bytes = 0;     // sub-chunk size (multiple of range_bytes)
  uint32_t range_bytes = 0, n_ranges = 0, slots = 0, evcap_words = 0;
  uint64_t max_records = 0;
  uint64_t row_cap = 0;       // RowDesc slots (rows one sub-chunk may emit)
  DevBuf recs, range_nrec, range_nlines, rec_base, line_base, events, dense, partial, stats1, row_desc, big_recs, tile_agg,
      tile_base, tile_partial, tile_scratch, slow;
  uint64_t scratch_cap = 0;   // bytes of tile blocks (grown on scratch_overflow)
  uint32_t slow_cap = 0;      // slow-path list entries (grown on slow_overflow)
};

struct Slot {
  cudaStream_t stream = nullptr;
  cudaEvent_t done = nullptr;
  DevBuf d_in, d_out, d_dosage, d_loci, d_loci_off, d_diags;
  DevBuf d_comp, d_blocks, d_fields, d_field_off, d_diag_starts;  // bgzf chunks; diagnostic fields
  Scratch sc;
  RunCounters *d_ctr = nullptr;
  RunCounters *h_ctr = nullptr;  // pinned
  uint8_t *h_out = nullptr;      // pinned
  size_t h_out_cap = 0;
  int8_t *h_dosage = nullptr;    // pinned
  size_t h_dosage_cap = 0;
  uint8_t *h_loci = nullptr;     // pinned
  size_t h_loci_cap = 0;
  uint64_t *h_loci_off = nullptr;  // pinned, rows + 1
  size_t h_loci_off_cap = 0;
  std::vector<bvcf_diag> h_diags;
  std::vector<uint32_t> h_diag_raw;
  bool busy = false;
  uint64_t seq = 0;
  const uint8_t *h_src = nullptr;
  size_t len = 0;
  uint32_t retries = 0;
  uint32_t diag_cap = 0;         // entries of d_diags the chunk was enqueued with
  // bgzf chunk: the text is inflate(comp) [0, text_len) then the tail; data lines start at `skip`
  bool bgzf = false;
  size_t skip = 0, text_len = 0, tail_len = 0;
  uint8_t *h_stage = nullptr;    // pinned: compressed bytes, block table, tail
  size_t h_stage_cap = 0;
  uint32_t *d_bad = nullptr;     // blocks that failed to inflate
  uint32_t *h_bad = nullptr;     // pinned copy
  std::vector<InflateBlock> blocks;
  std::vector<uint8_t> h_fields;
  std::vector<uint64_t> h_field_off, h_diag_starts;
};

constexpr uint32_t LOCI_GUESS = 32;          // first guess of locus bytes per row; the buffer grows to what a chunk reports
constexpr uint32_t DIAG_CAP0 = 1u << 16;   // first guess; grown to the count a chunk reports, then the chunk runs again

}  // namespace

struct bvcf_ctx {
  int device = 0;
  bvcf_config cfg{};
  std::string empty_field, field_delim;
  std::vector<std::string> allow, exclude;
  bool header_set = false;
  DevCfg dcfg{};
  DevBuf d_filt_blob, d_filt_off, d_names, d_name_off, d_name8, d_name16;
  std::vector<Slot> slots;
  // resident path
  DevBuf r_in, r_out, r_dosage, r_loci, r_loci_off, r_comp, r_blocks, r_def_slots, r_def_sizes, r_def_offs, r_def_out, r_diags;
  std::vector<bvcf_diag> r_h_diags;
  std::vector<int8_t> r_h_dosage;
  std::vector<uint8_t> r_h_loci;
  std::vector<uint64_t> r_h_loci_off;
  uint32_t *r_d_bad = nullptr;
  size_t r_in_bytes = 0;
  Scratch r_sc;
  cudaStream_t r_stream = nullptr;
  RunCounters *r_d_ctr = nullptr, *r_h_ctr = nullptr;
  std::vector<cudaEvent_t> ev_pool;
  double ev_factor = 0.5;  // event slice bytes per range byte
  uint32_t diag_cap = DIAG_CAP0;   // diagnostics a chunk may report (grown on demand, never truncated)
  uint32_t min_line_bytes = 16;    // line slots per range = range_bytes / max(H, this) + 2; halved on slot_overflow
  uint64_t launches = 0;
  std::string last_error;
  uint64_t r_last_records = 0;
  uint64_t r_last_len = 0;
};

namespace {

#define CK(call)                                                                          \
  do {                                                                                    \
    cudaError_t _e = (call);                                                              \
    if (_e != cudaSuccess) {                                                              \
      ctx->last_error = std::string(#call) + ": " + cudaGetErrorString(_e);               \
      return BVCF_E_CUDA;                                                                 \
    }                                                                                     \
  } while (0)

int dev_reserve(bvcf_ctx *ctx, DevBuf &b, size_t bytes) {
  if (bytes <= b.cap && b.p) return 0;
  if (b.p) cudaFree(b.p);
  b.p = nullptr;
  b.cap = 0;
  if (bytes == 0) bytes = 256;
  CK(cudaMalloc(&b.p, bytes));
  b.cap = bytes;
  return 0;
}
void dev_free(DevBuf &b) {
  if (b.p) cudaFree(b.p);
  b.p = nullptr;
  b.cap = 0;
}

uint64_t round_up(uint64_t v, uint64_t m) { return (v + m - 1) / m * m; }

// the scan kernel prefetches up to eight 512-byte windows past the last one it reads: allocated, never used
constexpr uint64_t IN_SLACK = 8192;

// choose the range size for `total` bytes: enough ranges to fill 148 SMs x 32 warps a few times over,
// large enough that re-reading one line per range boundary stays cheap
uint32_t choose_range_bytes(uint64_t total) {
  uint64_t r = total / (148ull * 32 * 3);
  r = round_up(std::max<uint64_t>(r, 1), 512);
  uint64_t cap_r = 256 * 1024;
  if (const char *e = getenv("BVCF_RANGE_KB")) cap_r = std::max(16, atoi(e)) * 1024ull;  // experiments
  r = std::min<uint64_t>(std::max<uint64_t>(r, 16 * 1024), cap_r);
  return (uint32_t)r;
}

int scratch_reserve(bvcf_ctx *ctx, Scratch &sc, uint64_t total_bytes, uint64_t sub_limit) {
  const int H = ctx->dcfg.H;
  sc.range_bytes = choose_range_bytes(total_bytes);
  // a record is scanned by the one warp that owns its start: with biobank-width lines (4+ bytes per sample)
  // ranges shorter than a line would leave most warps idle, so make a range hold at least ~1.25 lines
  {
    const uint64_t min_r = round_up(5ull * (uint64_t)std::max(ctx->dcfg.n_samples, 0), 512);
    if (min_r > sc.range_bytes) sc.range_bytes = (uint32_t)std::min<uint64_t>(min_r, 64ull << 20);
  }
  // sub-chunks of equal size (63 GB under a 24 GiB limit: three of 19.6 GiB, not two of 24 and a short one: the last
  // sub-chunk's kernels would run half empty)
  const uint64_t whole = round_up(total_bytes + 512, sc.range_bytes);
  const uint64_t n_sub = std::max<uint64_t>(1, (whole + sub_limit - 1) / std::max<uint64_t>(sub_limit, 1));
  uint64_t sub = std::min<uint64_t>(whole, round_up((whole + n_sub - 1) / n_sub, sc.range_bytes));
  sc.sub_bytes = sub;
  sc.n_ranges = (uint32_t)(sub / sc.range_bytes);
  // a record needs at least H bytes (H - 1 tabs + the newline); with H < 16 the first guess is 16 and slot_overflow
  // lowers it (bvcf_collect / bvcf_resident_run re-run the chunk)
  sc.slots = sc.range_bytes / std::max<uint32_t>((uint32_t)std::max(H, 1), ctx->min_line_bytes) + 2;
  uint64_t evb = (uint64_t)(sc.range_bytes * ctx->ev_factor) + 16 * 1024;
  if (ctx->dcfg.n_samples == 0) evb = 64;
  sc.evcap_words = (uint32_t)(evb / 4) & ~1u;  // quad events are 8-byte aligned
  while ((uint64_t)sc.n_ranges * sc.evcap_words >= (1ull << 32)) {  // event indices are 32-bit
    sc.n_ranges /= 2;
    sc.sub_bytes = (uint64_t)sc.n_ranges * sc.range_bytes;
  }
  sc.max_records = (uint64_t)sc.n_ranges * sc.slots;
  int rc;
  if ((rc = dev_reserve(ctx, sc.recs, sc.max_records * sizeof(LineRec)))) return rc;
  if ((rc = dev_reserve(ctx, sc.dense, sc.max_records * sizeof(LineRec)))) return rc;
  if ((rc = dev_reserve(ctx, sc.range_nrec, (size_t)sc.n_ranges * 4))) return rc;
  if ((rc = dev_reserve(ctx, sc.range_nlines, (size_t)sc.n_ranges * 4))) return rc;
  if ((rc = dev_reserve(ctx, sc.rec_base, (size_t)sc.n_ranges * 8))) return rc;
  if ((rc = dev_reserve(ctx, sc.line_base, (size_t)sc.n_ranges * 8))) return rc;
  if ((rc = dev_reserve(ctx, sc.events, (size_t)sc.n_ranges * sc.evcap_words * 4))) return rc;
  if ((rc = dev_reserve(ctx, sc.partial, 2 * PFX_BLOCKS * 8))) return rc;
  const uint64_t max_tiles = sc.max_records / TILE_THREADS + 2;
  if ((rc = dev_reserve(ctx, sc.tile_agg, max_tiles * sizeof(TileAgg)))) return rc;
  if ((rc = dev_reserve(ctx, sc.tile_base, max_tiles * sizeof(TileBase)))) return rc;
  if ((rc = dev_reserve(ctx, sc.tile_partial, (size_t)TSCAN_BLOCKS * TQ * 8))) return rc;
  // a tile's block: 1 KiB of per-record sizes, 32 bytes per row, the staged text (about 110 bytes per row)
  sc.scratch_cap = std::max<uint64_t>(sc.scratch_cap, std::min<uint64_t>(total_bytes / 8 + (8ull << 20), sc.max_records * 224ull + (1ull << 20)));
  if ((rc = dev_reserve(ctx, sc.tile_scratch, sc.scratch_cap + 64))) return rc;  // the copy-out reads whole words
  sc.slow_cap = std::max<uint32_t>(sc.slow_cap, 1u << 16);
  if ((rc = dev_reserve(ctx, sc.slow, (size_t)sc.slow_cap * sizeof(SlowRec)))) return rc;
  if (ctx->dcfg.n_samples > 0) {
    // rows queued for the names kernels: usually a third of the records; grown on row_overflow
    sc.row_cap = std::max<uint64_t>(sc.row_cap, sc.max_records / 2 + 1024);
    if ((rc = dev_reserve(ctx, sc.stats1, sc.max_records * sizeof(LineStats)))) return rc;
    if ((rc = dev_reserve(ctx, sc.row_desc, sc.row_cap * sizeof(RowDesc)))) return rc;
    if ((rc = dev_reserve(ctx, sc.big_recs, sc.max_records * 4))) return rc;
  }
  return 0;
}
void scratch_free(Scratch &sc) {
  for (DevBuf *b : {&sc.recs, &sc.range_nrec, &sc.range_nlines, &sc.rec_base, &sc.line_base, &sc.events, &sc.dense,
                    &sc.partial, &sc.stats1, &sc.row_desc, &sc.big_recs, &sc.tile_agg, &sc.tile_base, &sc.tile_partial,
                    &sc.tile_scratch, &sc.slow})
    dev_free(*b);
}

constexpr int N_STAGE_EV = 8;  // 0..5 stage boundaries, 6..7 inside the rows stage (compose | offsets | copy-out)
struct StageEvents {  // optional per-stage timing of one sub-chunk
  cudaEvent_t e[N_STAGE_EV];
};

// Enqueue the whole pipeline for data lines in [0, len) of d_in.  Never synchronises.
int enqueue_pipeline(bvcf_ctx *ctx, Scratch &sc, cudaStream_t st, const uint8_t *d_in, uint64_t begin, uint64_t len, uint64_t buf_len,
                     uint8_t *d_out, uint64_t out_cap, RunCounters *d_ctr, int8_t *d_dosage, uint64_t dosage_cap_rows,
                     uint8_t *d_loci, uint64_t loci_cap, unsigned long long *d_loci_off, uint32_t *d_diags,
                     uint32_t diag_cap, std::vector<StageEvents> *timing) {
  const DevCfg &dc = ctx->dcfg;
  // data lines live in [begin, len); ranges tile the region from begin rounded down to 512 bytes
  const uint64_t a0 = begin & ~511ull;
  const uint64_t total_ranges = (len - a0 + sc.range_bytes - 1) / sc.range_bytes;
  int smem = SCAN_WARPS * RING;
  if (const char *e = getenv("BVCF_SCAN_SMEM_KB")) smem = std::max(smem, atoi(e) * 1024);  // experiments: cap CTAs/SM
  cudaFuncSetAttribute(bvcf_scan_genotype_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  cudaFuncSetAttribute(bvcf_scan_genotype_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  int n_sm = 148;
  cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, ctx->device);
  for (uint64_t r0 = 0; r0 < total_ranges; r0 += sc.n_ranges) {
    const uint32_t nr = (uint32_t)std::min<uint64_t>(sc.n_ranges, total_ranges - r0);
    StageEvents *se = nullptr;
    if (timing) {
      timing->emplace_back();
      se = &timing->back();
      for (int i = 0; i < N_STAGE_EV; i++) {
        if (ctx->ev_pool.empty()) {
          cudaEvent_t e;
          CK(cudaEventCreate(&e));
          se->e[i] = e;
        } else {
          se->e[i] = ctx->ev_pool.back();
          ctx->ev_pool.pop_back();
        }
      }
      CK(cudaEventRecord(se->e[0], st));
    }
    // 1. scan: index + genotype events
    ScanParams sp{};
    sp.in = d_in; sp.begin = begin; sp.end = len; sp.buf_len = buf_len; sp.a0 = a0;
    sp.range_bytes = sc.range_bytes; sp.r0 = (uint32_t)r0; sp.n_ranges = nr;
    sp.slots_per_range = sc.slots; sp.evcap_words = sc.evcap_words;
    sp.recs = (LineRec *)sc.recs.p; sp.range_nrec = (uint32_t *)sc.range_nrec.p;
    sp.range_nlines = (uint32_t *)sc.range_nlines.p; sp.events = (uint32_t *)sc.events.p;
    sp.ctr = d_ctr; sp.H = dc.H; sp.eol_width = dc.eol_width;
    const unsigned grid = (nr + SCAN_WARPS - 1) / SCAN_WARPS;
    if (dc.n_samples > 0)
      bvcf_scan_genotype_kernel<true><<<grid, SCAN_WARPS * 32, smem, st>>>(sp);
    else
      bvcf_scan_genotype_kernel<false><<<grid, SCAN_WARPS * 32, smem, st>>>(sp);
    ctx->launches++;
    if (se) CK(cudaEventRecord(se->e[1], st));
    // 2. per-range counts -> bases
    PrefixParams pp{};
    pp.a = sp.range_nrec; pp.b = sp.range_nlines;
    pp.out_a = (uint64_t *)sc.rec_base.p; pp.out_b = (uint64_t *)sc.line_base.p;
    pp.partial = (unsigned long long *)sc.partial.p;
    pp.n_ptr = nullptr; pp.n_imm = nr; pp.ctr = d_ctr;
    bvcf_prefix_reduce_kernel<<<PFX_BLOCKS, PFX_THREADS, 0, st>>>(pp);
    bvcf_prefix_spine_kernel<<<1, 1024, 0, st>>>(pp);
    bvcf_prefix_scan_kernel<<<PFX_BLOCKS, PFX_THREADS, 0, st>>>(pp);
    // 3. compaction
    CompactParams cp{};
    cp.recs = sp.recs; cp.range_nrec = sp.range_nrec; cp.rec_base = pp.out_a; cp.line_base = pp.out_b;
    cp.dense = (LineRec *)sc.dense.p; cp.n_ranges = nr; cp.slots_per_range = sc.slots; cp.evcap_words = sc.evcap_words;
    bvcf_compact_lines_kernel<<<(nr + 7) / 8, 256, 0, st>>>(cp);
    ctx->launches += 4;
    if (se) CK(cudaEventRecord(se->e[2], st));
    // many more CTAs than SMs: each warp gets about one block of 32 records/rows and the hardware
    // scheduler evens out the very different row sizes (1 .. 2,500 names)
    const unsigned wgrid = (unsigned)n_sm * 64;
    // 3b. ALT #1 genotype summary per record (warp per record)
    if (dc.n_samples > 0) {
      StatsParams tp{};
      tp.in = d_in; tp.cfg = dc; tp.lines = cp.dense; tp.events = sp.events; tp.stats = (LineStats *)sc.stats1.p; tp.ctr = d_ctr;
      tp.big_recs = (uint32_t *)sc.big_recs.p;
      bvcf_line_stats_kernel<<<wgrid, 256, 0, st>>>(tp);
      bvcf_line_stats_big_kernel<<<(unsigned)n_sm * 4, 256, 0, st>>>(tp);
      ctx->launches += 2;
    }
    if (se) CK(cudaEventRecord(se->e[3], st));
    // 4. rows: FILTER + getAlleles + row text + short name lists, one pass (tile of 128 records per CTA)
    static const bool no_vec = getenv("BVCF_NO_NAMES_VEC") != nullptr;  // experiments
    const bool vec = (dc.name8 || dc.name16) && dc.want_tsv && !no_vec && dc.n_samples > 0;
    TileParams tp{};
    tp.in = d_in; tp.cfg = dc; tp.lines = cp.dense; tp.events = sp.events; tp.stats = (const LineStats *)sc.stats1.p;
    tp.out = d_out; tp.out_cap = out_cap; tp.ctr = d_ctr;
    tp.tile_agg = (TileAgg *)sc.tile_agg.p; tp.tile_base = (TileBase *)sc.tile_base.p;
    tp.tile_partial = (unsigned long long *)sc.tile_partial.p;
    tp.scratch = (uint8_t *)sc.tile_scratch.p; tp.scratch_cap = sc.scratch_cap;
    tp.slow = (SlowRec *)sc.slow.p; tp.slow_cap = sc.slow_cap;
    tp.row_desc = (RowDesc *)sc.row_desc.p; tp.row_desc_cap = dc.n_samples > 0 ? sc.row_cap : 0;
    tp.long_words = vec ? 8192u : 0u;  // rows beyond 4,096 quads: a CTA per row
    {
      // rows of up to 16 quads: a lane per row.  Measured on 600,000 chr1-shape variants (names stage): no mid class
      // 0.349 ms, 16 quads 0.345, 32 quads 0.359, 64 quads 0.408, 128 quads 0.49 -- a lane's own event list and its
      // scattered 8-byte stores cost more than the idle lanes of a warp-per-row sweep once rows hold a few dozen names
      static const int mid_q = getenv("BVCF_MID_QUADS") ? atoi(getenv("BVCF_MID_QUADS")) : 16;  // experiments
      tp.mid_words = (dc.want_tsv && dc.n_samples > 0) ? 2u * (uint32_t)std::max(mid_q, 0) : 0u;
      if (!vec) tp.mid_words = 0;  // names_big_kernel serves every list
    }
    tp.dosage = d_dosage; tp.dosage_cap_rows = dosage_cap_rows;
    tp.loci = d_loci; tp.loci_cap = loci_cap; tp.loci_off = d_loci_off;
    tp.diag.diags = d_diags; tp.diag.cap = diag_cap; tp.diag.ctr = d_ctr;
    {
      auto launch = [&](auto kern, uint32_t arena, uint32_t rows, int minb) {
        const uint32_t smem = TILE_WARPS * tile_smem_warp(arena, rows);
        cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        kern<<<(unsigned)n_sm * minb, TILE_WARPS * 32, smem, st>>>(tp);
      };
      // (5, 6 and 8 resident CTAs per SM were measured too: the spills of a 96 / 80 / 64-register build cost more than
      // the extra warps hide -- rows 0.42 -> 0.51 / 0.52 / 0.55 ms on 600,000 chr1-shape variants)
      // L2 prefetch of the next tile's lines / scratch block: measured, no gain (compose 0.323 -> 0.329 ms, copy-out
      // 0.116 -> 0.124 ms on 600,000 chr1-shape variants: the waits are dependent L1/L2 hits, not DRAM), so off
      static const int pf = getenv("BVCF_PREFETCH") ? atoi(getenv("BVCF_PREFETCH")) : 0;  // experiments: bit 0 compose, bit 1 copy-out
      static const bool sites_old = getenv("BVCF_SITES_OLD") != nullptr;  // experiments: the thread-per-record composer
      if (dc.n_samples == 0 && !sites_old) {
        static const int sv = getenv("BVCF_SITES_VAR") ? atoi(getenv("BVCF_SITES_VAR")) : 0;  // experiments
        // 8 resident CTAs (64 registers, 3.5 KiB arena + 96 rows per warp) against 5 (80 registers, 6 KiB + 128 rows):
        // 19.5 against 23.3 ms on 50 M lines -- the kernel waits on dependent loads and taken branches, warps hide both
        // (REF / ALT held in registers, which pays at 128 registers, spills at 64: 20.3 ms; 7 CTAs x 72 registers with
        // them: 20.9 ms; 8 CTAs without: 19.5 ms)
        if (sv == 5) launch(bvcf_compose_sites_kernel<5, 6144, 128, true>, 6144, 128, 5);
        else launch(bvcf_compose_sites_kernel<8, 3584, 96, false>, 3584, 96, 8);
      } else if (dc.n_samples == 0) {
        if (pf & 1) launch(bvcf_compose_kernel<4, 8192, 160, true>, 8192, 160, 4);
        else launch(bvcf_compose_kernel<4, 8192, 160, false>, 8192, 160, 4);
      } else {
        // the build for the default flags: TSV rows, no --keepPos/Id/Info, no dosage matrix, 7-character names joined by
        // one character -- a smaller kernel (see "Code size" in DESIGN.md)
        static const bool no_spec = getenv("BVCF_NO_SPEC") != nullptr;  // experiments
        const bool spec = !no_spec && dc.want_tsv && !dc.keep_pos && !dc.keep_id && !dc.keep_info && !dc.want_dosage && dc.name8 &&
                          dc.delim_len == 1 && dc.name_fixed_w == 7;
        if (pf & 1) launch(bvcf_compose_kernel<4, 10240, 48, true>, 10240, 48, 4);
        else if (spec) launch(bvcf_compose_kernel<4, 10240, 48, false, true>, 10240, 48, 4);
        else launch(bvcf_compose_kernel<4, 10240, 48, false>, 10240, 48, 4);
      }
      if (se) CK(cudaEventRecord(se->e[6], st));
      bvcf_tile_reduce_kernel<<<TSCAN_BLOCKS, TSCAN_THREADS, 0, st>>>(tp);
      bvcf_tile_spine_kernel<<<1, 32, 0, st>>>(tp);
      bvcf_tile_offsets_kernel<<<TSCAN_BLOCKS, TSCAN_THREADS, 0, st>>>(tp);
      if (se) CK(cudaEventRecord(se->e[7], st));
      if (dc.want_dosage && dc.n_samples > 0 && d_dosage) {
        bvcf_dosage_zero_kernel<<<(unsigned)n_sm * 8, 256, 0, st>>>(tp);
        ctx->launches += 1;
      }
      if (pf & 2) bvcf_copyout_kernel<true><<<(unsigned)n_sm * 16, TILE_WARPS * 32, 0, st>>>(tp);
      else bvcf_copyout_kernel<false><<<(unsigned)n_sm * 16, TILE_WARPS * 32, 0, st>>>(tp);
    }
    bvcf_slow_rows_kernel<<<(unsigned)n_sm, 64, 0, st>>>(tp);
    ctx->launches += 6;
    if (se) CK(cudaEventRecord(se->e[4], st));
    // 5. long sample-name lists + their dosage rows: a warp per queued row -- as aligned vectors when every list
    // item has one size of 5..16 bytes (bvcf_names.cuh) -- and a CTA per row beyond 4,096 quads
    if (dc.n_samples > 0) {
      NamesParams np{};
      np.in = d_in; np.cfg = dc; np.lines = cp.dense; np.events = sp.events; np.row_desc = (const RowDesc *)sc.row_desc.p;
      np.row_desc_cap = sc.row_cap; np.out = d_out; np.ctr = d_ctr; np.dosage = d_dosage; np.dosage_cap_rows = dosage_cap_rows;
      np.long_words = tp.long_words;
      if (vec) {
        const unsigned g1 = (unsigned)n_sm * 18, g2 = (unsigned)n_sm * 2;
        const bool dos = dc.want_dosage && d_dosage;
        if (tp.mid_words) {
          if (dos) bvcf_names_mid_kernel<true><<<(unsigned)n_sm * 16, 128, 0, st>>>(np);
          else bvcf_names_mid_kernel<false><<<(unsigned)n_sm * 16, 128, 0, st>>>(np);
          ctx->launches++;
        }
        if (dc.n_samples <= 65000) {
          if (dos) {
            bvcf_names_vec_kernel<uint16_t, true><<<g1, NVEC_WARPS * 32, 0, st>>>(np);
            bvcf_names_long_kernel<uint16_t, true><<<g2, NLONG_WARPS * 32, 0, st>>>(np);
          } else {
            bvcf_names_vec_kernel<uint16_t, false><<<g1, NVEC_WARPS * 32, 0, st>>>(np);
            bvcf_names_long_kernel<uint16_t, false><<<g2, NLONG_WARPS * 32, 0, st>>>(np);
          }
        } else {
          if (dos) {
            bvcf_names_vec_kernel<uint32_t, true><<<g1, NVEC_WARPS * 32, 0, st>>>(np);
            bvcf_names_long_kernel<uint32_t, true><<<g2, NLONG_WARPS * 32, 0, st>>>(np);
          } else {
            bvcf_names_vec_kernel<uint32_t, false><<<g1, NVEC_WARPS * 32, 0, st>>>(np);
            bvcf_names_long_kernel<uint32_t, false><<<g2, NLONG_WARPS * 32, 0, st>>>(np);
          }
        }
        ctx->launches += 2;
      } else {
        bvcf_names_big_kernel<<<wgrid * 4, NAMES_WARPS * 32, 0, st>>>(np);
        ctx->launches++;
      }
    }
    if (se) CK(cudaEventRecord(se->e[5], st));
  }
  CK(cudaGetLastError());
  return 0;
}

void fill_dcfg(bvcf_ctx *ctx) {
  DevCfg &d = ctx->dcfg;
  const bvcf_config &c = ctx->cfg;
  d.eol_width = c.eol_width == 2 ? 2 : 1;
  d.keep_id = c.keep_id != 0; d.keep_info = c.keep_info != 0; d.keep_pos = c.keep_pos != 0;
  d.want_tsv = c.want_tsv != 0; d.want_dosage = c.want_dosage != 0;
  d.allow_all = c.n_allow < 0;
  d.n_allow = c.n_allow < 0 ? 0 : (int)ctx->allow.size();
  d.n_excl = (int)ctx->exclude.size();
  d.empty_len = (int)ctx->empty_field.size();
  memcpy(d.empty, ctx->empty_field.data(), ctx->empty_field.size());
  d.delim_len = (int)ctx->field_delim.size();
  memcpy(d.delim, ctx->field_delim.data(), ctx->field_delim.size());
  {  // main.go:612-616,634-637,648-651,667 with no samples: three empty lists with ratio 0, then ac, an, sampleMaf = 0
    std::string t;
    for (int k = 0; k < 3; k++) t += ctx->empty_field + "\t0\t";
    t += "0\t0\t0";
    d.tail0_len = (int)t.size();
    memcpy(d.tail0, t.data(), t.size());
  }
}

Slot *find_slot(bvcf_ctx *ctx, uint64_t seq) {
  for (auto &s : ctx->slots)
    if (s.busy && s.seq == seq) return &s;
  return nullptr;
}

// device diagnostics (DIAG_WORDS words each, in the order the threads pushed them) -> bvcf_diag sorted by line, then
// ALT number: an 8-byte key per entry is sorted, not the 32-byte records
void decode_diags(const uint32_t *raw, uint32_t nd, std::vector<bvcf_diag> &out) {
  out.clear();
  if (!nd) return;
  std::vector<std::pair<uint64_t, uint32_t>> key(nd);
  uint64_t lo = ~0ull;
  for (uint32_t i = 0; i < nd; i++) {
    const uint32_t *w = raw + (size_t)DIAG_WORDS * i;
    lo = std::min(lo, (uint64_t)w[0] | ((uint64_t)w[1] << 32));
  }
  bool packed = true;  // (line - first line) and the ALT number share 64 bits: 40 + 24
  for (uint32_t i = 0; i < nd; i++) {
    const uint32_t *w = raw + (size_t)DIAG_WORDS * i;
    const uint64_t ln = ((uint64_t)w[0] | ((uint64_t)w[1] << 32)) - lo;
    if (ln >= (1ull << 40) || w[2] >= (1u << 24)) { packed = false; break; }
    key[i] = {(ln << 24) | w[2], i};
  }
  out.resize(nd);
  auto fill = [&](uint32_t dst, uint32_t src) {
    const uint32_t *w = raw + (size_t)DIAG_WORDS * src;
    bvcf_diag d;
    d.line_no = (uint64_t)w[0] | ((uint64_t)w[1] << 32);
    d.alt_no = (int32_t)w[2];
    d.code = (int32_t)w[3];
    d.line_start = (uint64_t)w[4] | ((uint64_t)w[5] << 32);
    out[dst] = d;
  };
  if (packed) {
    std::sort(key.begin(), key.end());
    for (uint32_t i = 0; i < nd; i++) fill(i, key[i].second);
  } else {
    for (uint32_t i = 0; i < nd; i++) fill(i, i);
    std::sort(out.begin(), out.end(), [](const bvcf_diag &a, const bvcf_diag &b) {
      return a.line_no != b.line_no ? a.line_no < b.line_no : a.alt_no < b.alt_no;
    });
  }
}

// A bgzf chunk's compressed bytes, block table and tail are in the slot's pinned staging buffer: upload them, inflate the
// blocks into d_in, put the tail after the text.  Only the first attempt does this -- a retry finds the text on the device.
int slot_inflate(bvcf_ctx *ctx, Slot &s, size_t comp_len) {
  const size_t nb = s.blocks.size(), tab_off = round_up(comp_len, 16), tail_off = tab_off + nb * sizeof(InflateBlock);
  int rc;
  if ((rc = dev_reserve(ctx, s.d_comp, comp_len + 16))) return rc;  // the bit reader may look 11 bytes past the payload
  if ((rc = dev_reserve(ctx, s.d_blocks, nb * sizeof(InflateBlock)))) return rc;
  if (!s.d_bad) CK(cudaMalloc(&s.d_bad, 4));
  if (!s.h_bad) CK(cudaMallocHost(&s.h_bad, 8));  // [0] bad blocks, [1] last text byte
  s.h_bad[0] = s.h_bad[1] = 0;
  CK(cudaMemsetAsync(s.d_bad, 0, 4, s.stream));
  if (nb) {
    CK(cudaMemcpyAsync(s.d_comp.p, s.h_stage, comp_len, cudaMemcpyHostToDevice, s.stream));
    CK(cudaMemcpyAsync(s.d_blocks.p, s.h_stage + tab_off, nb * sizeof(InflateBlock), cudaMemcpyHostToDevice, s.stream));
    InflateParams ip{};
    ip.comp = (const uint8_t *)s.d_comp.p; ip.out = (uint8_t *)s.d_in.p; ip.blocks = (const InflateBlock *)s.d_blocks.p;
    ip.n_blocks = (uint32_t)nb; ip.n_bad = s.d_bad;
    cudaFuncSetAttribute(bvcf_inflate_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)INF_SMEM);
    bvcf_inflate_kernel<<<ip.n_blocks, 32, INF_SMEM, s.stream>>>(ip);
    ctx->launches++;
  }
  if (s.tail_len)
    CK(cudaMemcpyAsync((uint8_t *)s.d_in.p + s.text_len, s.h_stage + tail_off, s.tail_len, cudaMemcpyHostToDevice, s.stream));
  CK(cudaMemcpyAsync(s.h_bad, s.d_bad, 4, cudaMemcpyDeviceToHost, s.stream));
  if (s.len > s.skip && !s.tail_len)  // the text must end with a newline: its last byte, for bvcf_collect
    CK(cudaMemcpyAsync(s.h_bad + 1, (const uint8_t *)s.d_in.p + s.len - 1, 1, cudaMemcpyDeviceToHost, s.stream));
  else
    s.h_bad[1] = '\n';
  return 0;
}

int slot_enqueue(bvcf_ctx *ctx, Slot &s, bool upload, size_t comp_len = 0) {
  const uint64_t len = s.len;
  const uint64_t buf_len = round_up(len, 1024) + 2048;
  int rc;
  if ((rc = dev_reserve(ctx, s.d_in, buf_len + IN_SLACK))) return rc;
  if ((rc = scratch_reserve(ctx, s.sc, len - (s.skip & ~511ull), ctx->cfg.resident_subchunk_bytes))) return rc;
  if (s.d_out.cap == 0) {
    if ((rc = dev_reserve(ctx, s.d_out, std::max<size_t>(len / 2, 1 << 20)))) return rc;
  }
  const DevCfg &dc = ctx->dcfg;
  uint64_t dos_rows = 0;
  if (dc.want_dosage && dc.n_samples > 0) {
    dos_rows = std::min<uint64_t>(s.d_dosage.cap / (uint64_t)dc.n_samples, s.d_loci_off.cap / 8);
    if (dos_rows == 0) {
      const uint64_t est = std::max<uint64_t>(len / std::max(1, dc.H) * 2, 1024);
      if ((rc = dev_reserve(ctx, s.d_dosage, est * dc.n_samples))) return rc;
      if ((rc = dev_reserve(ctx, s.d_loci_off, est * 8))) return rc;
      if ((rc = dev_reserve(ctx, s.d_loci, est * LOCI_GUESS))) return rc;
      dos_rows = est;
    }
  }
  s.diag_cap = ctx->diag_cap;
  if ((rc = dev_reserve(ctx, s.d_diags, (size_t)s.diag_cap * DIAG_WORDS * 4))) return rc;
  if (upload && s.bgzf) {
    if ((rc = slot_inflate(ctx, s, comp_len))) return rc;
  } else if (upload) {
    CK(cudaMemcpyAsync(s.d_in.p, s.h_src, len, cudaMemcpyHostToDevice, s.stream));
  }
  CK(cudaMemsetAsync((uint8_t *)s.d_in.p + len, '\n', buf_len - len, s.stream));
  CK(cudaMemsetAsync(s.d_ctr, 0, sizeof(RunCounters), s.stream));
  rc = enqueue_pipeline(ctx, s.sc, s.stream, (const uint8_t *)s.d_in.p, s.skip, len, buf_len, (uint8_t *)s.d_out.p, s.d_out.cap,
                        s.d_ctr, (int8_t *)s.d_dosage.p, dos_rows, (uint8_t *)s.d_loci.p, s.d_loci.cap,
                        (unsigned long long *)s.d_loci_off.p, (uint32_t *)s.d_diags.p, s.diag_cap, nullptr);
  if (rc) return rc;
  CK(cudaMemcpyAsync(s.h_ctr, s.d_ctr, sizeof(RunCounters), cudaMemcpyDeviceToHost, s.stream));
  CK(cudaEventRecord(s.done, s.stream));
  return 0;
}

}  // namespace

// ---------------------------------------------------------------------------------------------------
extern "C" {

int bvcf_abi_version(void) { return BVCF_ABI_VERSION; }

const char *bvcf_strerror(int rc) {
  switch (rc) {
    case BVCF_OK: return "ok";
    case BVCF_E_ARG: return "bad argument";
    case BVCF_E_CUDA: return "CUDA error (see bvcf_last_error)";
    case BVCF_E_STATE: return "bad call order or no free slot";
    case BVCF_E_NOT_ALIGNED: return "chunk does not end with a newline";
    case BVCF_E_TOO_LARGE: return "input exceeds a library limit";
    case BVCF_E_NOMEM: return "out of host memory";
    default: return "unknown error";
  }
}

const char *bvcf_last_error(const bvcf_ctx *ctx) { return ctx ? ctx->last_error.c_str() : ""; }
uint64_t bvcf_launch_count(const bvcf_ctx *ctx) { return ctx ? ctx->launches : 0; }

int bvcf_header_line(const bvcf_config *cfg, char *buf, size_t cap) {
  // parse.Header + optional columns (main.go:219-239)
  std::string h =
      "chrom\tpos\ttype\tref\talt\ttrTv\theterozygotes\theterozygosity\thomozygotes\thomozygosity\tmissingGenos\t"
      "missingness\tac\tan\tsampleMaf";
  if (cfg && cfg->keep_pos) h += "\tvcfPos";
  if (cfg && cfg->keep_id) h += "\tid";
  if (cfg && cfg->keep_info) h += "\talleleIdx\tinfo";
  if (buf && cap) {
    const size_t n = std::min(cap - 1, h.size());
    memcpy(buf, h.data(), n);
    buf[n] = 0;
  }
  return (int)h.size();
}

int bvcf_create(bvcf_ctx **out, int cuda_device, const bvcf_config *cfg) {
  if (!out || !cfg) return BVCF_E_ARG;
  *out = nullptr;
  bvcf_ctx *ctx = new (std::nothrow) bvcf_ctx();
  if (!ctx) return BVCF_E_NOMEM;
  ctx->device = cuda_device;
  ctx->cfg = *cfg;
  ctx->empty_field = cfg->empty_field ? cfg->empty_field : "!";
  ctx->field_delim = cfg->field_delim ? cfg->field_delim : ";";
  if (ctx->empty_field.size() > 63 || ctx->field_delim.size() > 63) { delete ctx; return BVCF_E_TOO_LARGE; }
  for (int i = 0; i < cfg->n_allow; i++) ctx->allow.push_back(cfg->allow[i] ? cfg->allow[i] : "");
  for (int i = 0; i < cfg->n_exclude; i++) ctx->exclude.push_back(cfg->exclude[i] ? cfg->exclude[i] : "");
  if (ctx->allow.size() + ctx->exclude.size() > 64) { delete ctx; return BVCF_E_TOO_LARGE; }
  if (const char *e = getenv("BVCF_DIAG_CAP")) ctx->diag_cap = (uint32_t)std::max(1, atoi(e));  // tests: force the grow-and-retry path
  if (ctx->cfg.n_slots <= 0) ctx->cfg.n_slots = 3;
  if (ctx->cfg.max_chunk_bytes == 0) ctx->cfg.max_chunk_bytes = 256ull << 20;
  if (ctx->cfg.resident_subchunk_bytes == 0) ctx->cfg.resident_subchunk_bytes = 24ull << 30;
  ctx->cfg.allow = nullptr; ctx->cfg.exclude = nullptr; ctx->cfg.empty_field = nullptr; ctx->cfg.field_delim = nullptr;

  auto fail = [&](int rc) { *out = ctx; bvcf_destroy(ctx); *out = nullptr; return rc; };
  // no CPU fallback: a missing device is an error
  int n_dev = 0;
  cudaError_t e = cudaGetDeviceCount(&n_dev);
  if (e != cudaSuccess || cuda_device < 0 || cuda_device >= n_dev) {
    fprintf(stderr, "libbvcf: no usable CUDA device %d (%s)\n", cuda_device,
            e != cudaSuccess ? cudaGetErrorString(e) : "index out of range");
    delete ctx;
    return BVCF_E_CUDA;
  }
  if (cudaSetDevice(cuda_device) != cudaSuccess) { delete ctx; return BVCF_E_CUDA; }

  // FILTER table
  std::vector<uint8_t> blob;
  std::vector<uint32_t> off{0};
  for (auto &s : ctx->allow) { blob.insert(blob.end(), s.begin(), s.end()); off.push_back((uint32_t)blob.size()); }
  for (auto &s : ctx->exclude) { blob.insert(blob.end(), s.begin(), s.end()); off.push_back((uint32_t)blob.size()); }
  if (blob.size() > FILT_SMEM) return fail(BVCF_E_TOO_LARGE);
  if (dev_reserve(ctx, ctx->d_filt_blob, blob.size() + 16)) return fail(BVCF_E_CUDA);
  if (dev_reserve(ctx, ctx->d_filt_off, off.size() * 4)) return fail(BVCF_E_CUDA);
  if (!blob.empty()) cudaMemcpy(ctx->d_filt_blob.p, blob.data(), blob.size(), cudaMemcpyHostToDevice);
  cudaMemcpy(ctx->d_filt_off.p, off.data(), off.size() * 4, cudaMemcpyHostToDevice);
  ctx->dcfg.filt_blob = (const uint8_t *)ctx->d_filt_blob.p;
  ctx->dcfg.filt_off = (const uint32_t *)ctx->d_filt_off.p;
  ctx->dcfg.filt_bytes = (int)blob.size();
  fill_dcfg(ctx);

  ctx->slots.resize(ctx->cfg.n_slots);
  for (auto &s : ctx->slots) {
    if (cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking) != cudaSuccess) return fail(BVCF_E_CUDA);
    if (cudaEventCreateWithFlags(&s.done, cudaEventDisableTiming) != cudaSuccess) return fail(BVCF_E_CUDA);
    if (cudaMalloc(&s.d_ctr, sizeof(RunCounters)) != cudaSuccess) return fail(BVCF_E_CUDA);
    if (cudaMallocHost(&s.h_ctr, sizeof(RunCounters)) != cudaSuccess) return fail(BVCF_E_CUDA);
  }
  if (cudaStreamCreateWithFlags(&ctx->r_stream, cudaStreamNonBlocking) != cudaSuccess) return fail(BVCF_E_CUDA);
  if (cudaMalloc(&ctx->r_d_ctr, sizeof(RunCounters)) != cudaSuccess) return fail(BVCF_E_CUDA);
  if (cudaMallocHost(&ctx->r_h_ctr, sizeof(RunCounters)) != cudaSuccess) return fail(BVCF_E_CUDA);
  *out = ctx;
  return BVCF_OK;
}

void bvcf_destroy(bvcf_ctx *ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaDeviceSynchronize();
  for (auto &s : ctx->slots) {
    if (s.stream) cudaStreamDestroy(s.stream);
    if (s.done) cudaEventDestroy(s.done);
    for (DevBuf *b : {&s.d_in, &s.d_out, &s.d_dosage, &s.d_loci, &s.d_loci_off, &s.d_diags, &s.d_comp, &s.d_blocks, &s.d_fields,
                      &s.d_field_off, &s.d_diag_starts})
      dev_free(*b);
    if (s.d_bad) cudaFree(s.d_bad);
    if (s.h_bad) cudaFreeHost(s.h_bad);
    if (s.h_stage) cudaFreeHost(s.h_stage);
    scratch_free(s.sc);
    if (s.d_ctr) cudaFree(s.d_ctr);
    if (s.h_ctr) cudaFreeHost(s.h_ctr);
    if (s.h_out) cudaFreeHost(s.h_out);
    if (s.h_dosage) cudaFreeHost(s.h_dosage);
    if (s.h_loci) cudaFreeHost(s.h_loci);
    if (s.h_loci_off) cudaFreeHost(s.h_loci_off);
  }
  for (DevBuf *b : {&ctx->d_filt_blob, &ctx->d_filt_off, &ctx->d_names, &ctx->d_name_off, &ctx->d_name8, &ctx->d_name16, &ctx->r_in, &ctx->r_out,
                    &ctx->r_dosage, &ctx->r_loci, &ctx->r_loci_off, &ctx->r_comp, &ctx->r_blocks, &ctx->r_def_slots,
                    &ctx->r_def_sizes, &ctx->r_def_offs, &ctx->r_def_out, &ctx->r_diags})
    dev_free(*b);
  scratch_free(ctx->r_sc);
  if (ctx->r_stream) cudaStreamDestroy(ctx->r_stream);
  if (ctx->r_d_ctr) cudaFree(ctx->r_d_ctr);
  if (ctx->r_d_bad) cudaFree(ctx->r_d_bad);
  if (ctx->r_h_ctr) cudaFreeHost(ctx->r_h_ctr);
  for (auto e : ctx->ev_pool) cudaEventDestroy(e);
  delete ctx;
}

int bvcf_set_header(bvcf_ctx *ctx, const char *chrom_line, size_t len) {
  if (!ctx || !chrom_line) return BVCF_E_ARG;
  cudaSetDevice(ctx->device);
  while (len && (chrom_line[len - 1] == '\n' || chrom_line[len - 1] == '\r')) len--;  // chomp (main.go:281)
  std::vector<std::string> f;
  size_t s = 0;
  for (size_t i = 0; i <= len; i++) {
    if (i == len || chrom_line[i] == '\t') { f.emplace_back(chrom_line + s, i - s); s = i + 1; }
  }
  const int H = (int)f.size();
  if (H < 8) return BVCF_E_ARG;  // the reference would panic indexing FILTER/INFO
  const int ns = H > 9 ? H - 9 : 0;  // main.go:505-509
  if ((uint32_t)ns > MAX_SAMPLES) return BVCF_E_TOO_LARGE;
  std::vector<uint8_t> blob;
  std::vector<uint32_t> off{0};
  int fixed_w = -1;
  for (int i = 0; i < ns; i++) {
    std::string nm = f[9 + i];
    if (ctx->cfg.normalize_dots)
      for (auto &c : nm) if (c == '.') c = '_';  // parse.NormalizeHeader (main.go:296)
    blob.insert(blob.end(), nm.begin(), nm.end());
    off.push_back((uint32_t)blob.size());
    if (i == 0) fixed_w = (int)nm.size();
    else if (fixed_w != (int)nm.size()) fixed_w = 0;
  }
  if (fixed_w < 0) fixed_w = 0;
  int rc;
  if ((rc = dev_reserve(ctx, ctx->d_names, blob.size() + 16))) return rc;
  if ((rc = dev_reserve(ctx, ctx->d_name_off, off.size() * 4))) return rc;
  if (!blob.empty()) CK(cudaMemcpy(ctx->d_names.p, blob.data(), blob.size(), cudaMemcpyHostToDevice));
  CK(cudaMemcpy(ctx->d_name_off.p, off.data(), off.size() * 4, cudaMemcpyHostToDevice));
  ctx->dcfg.H = H;
  ctx->dcfg.n_samples = ns;
  ctx->dcfg.names = (const uint8_t *)ctx->d_names.p;
  ctx->dcfg.name_off = (const uint32_t *)ctx->d_name_off.p;
  ctx->dcfg.name_fixed_w = fixed_w;
  ctx->dcfg.name8 = nullptr;
  ctx->dcfg.name16 = nullptr;
  ctx->dcfg.item_bytes = 0;
  if (fixed_w == 7 && ctx->field_delim.size() == 1 && ns > 0) {
    std::vector<unsigned long long> n8(ns);
    for (int i = 0; i < ns; i++) {
      unsigned long long v = 0;
      for (int k = 0; k < 7; k++) v |= (unsigned long long)blob[(size_t)i * 7 + k] << (8 * k);
      v |= (unsigned long long)(uint8_t)ctx->field_delim[0] << 56;
      n8[i] = v;
    }
    if ((rc = dev_reserve(ctx, ctx->d_name8, n8.size() * 8))) return rc;
    CK(cudaMemcpy(ctx->d_name8.p, n8.data(), n8.size() * 8, cudaMemcpyHostToDevice));
    ctx->dcfg.name8 = (const unsigned long long *)ctx->d_name8.p;
    ctx->dcfg.item_bytes = 8;
  } else if (fixed_w > 0 && ns > 0 && fixed_w + (int)ctx->field_delim.size() >= 5 && fixed_w + (int)ctx->field_delim.size() <= 16) {
    // any other fixed width: 16-byte padded items for the vector names kernels
    const int I = fixed_w + (int)ctx->field_delim.size();
    std::vector<uint8_t> n16((size_t)ns * 16, 0);
    for (int i = 0; i < ns; i++) {
      memcpy(&n16[(size_t)i * 16], &blob[(size_t)i * fixed_w], fixed_w);
      memcpy(&n16[(size_t)i * 16 + fixed_w], ctx->field_delim.data(), ctx->field_delim.size());
    }
    if ((rc = dev_reserve(ctx, ctx->d_name16, n16.size()))) return rc;
    CK(cudaMemcpy(ctx->d_name16.p, n16.data(), n16.size(), cudaMemcpyHostToDevice));
    ctx->dcfg.name16 = (const uint4 *)ctx->d_name16.p;
    ctx->dcfg.item_bytes = I;
  }
  ctx->header_set = true;
  return BVCF_OK;
}

int bvcf_host_alloc(void **ptr, size_t bytes) {
  if (!ptr) return BVCF_E_ARG;
  return cudaMallocHost(ptr, bytes ? bytes : 1) == cudaSuccess ? BVCF_OK : BVCF_E_CUDA;
}
void bvcf_host_free(void *ptr) {
  if (ptr) cudaFreeHost(ptr);
}

int bvcf_submit(bvcf_ctx *ctx, uint64_t seq, const uint8_t *chunk, size_t len) {
  if (!ctx || (!chunk && len)) return BVCF_E_ARG;
  if (!ctx->header_set) return BVCF_E_STATE;
  if (len > ctx->cfg.max_chunk_bytes || len >= (1ull << 31)) return BVCF_E_TOO_LARGE;
  if (len && chunk[len - 1] != '\n') return BVCF_E_NOT_ALIGNED;
  if (find_slot(ctx, seq)) return BVCF_E_STATE;
  Slot *s = nullptr;
  for (auto &x : ctx->slots)
    if (!x.busy) { s = &x; break; }
  if (!s) return BVCF_E_STATE;
  cudaSetDevice(ctx->device);
  s->busy = true; s->seq = seq; s->h_src = chunk; s->len = len; s->retries = 0;
  s->bgzf = false; s->skip = 0; s->text_len = len; s->tail_len = 0;
  const int rc = slot_enqueue(ctx, *s, true);
  if (rc) s->busy = false;
  return rc;
}

int bvcf_collect(bvcf_ctx *ctx, uint64_t seq, const uint8_t **tsv, size_t *tsv_len, bvcf_dosage_batch *dosage,
                 const bvcf_diag **diags, size_t *n_diags, bvcf_chunk_stats *stats) {
  if (!ctx) return BVCF_E_ARG;
  Slot *s = find_slot(ctx, seq);
  if (!s) return BVCF_E_STATE;
  cudaSetDevice(ctx->device);
  ctx->last_error.clear();
  const DevCfg &dc = ctx->dcfg;
  static const bool trace = getenv("BVCF_TRACE") != nullptr;  // experiments: where a collect spends its time
  const auto t_begin = std::chrono::steady_clock::now();
  for (;;) {
    CK(cudaEventSynchronize(s->done));
    if (s->bgzf && s->h_bad[0]) {  // a corrupt member: whatever the pipeline made of its text is not looked at
      ctx->last_error = std::to_string(s->h_bad[0]) + " bgzf block(s) failed to inflate or failed their CRC-32 / ISIZE check";
      return BVCF_E_ARG;
    }
    if (s->bgzf && s->len > s->skip && (s->h_bad[1] & 0xFFu) != '\n') return BVCF_E_NOT_ALIGNED;
    const RunCounters &c = *s->h_ctr;
    bool again = false;
    if (c.slot_overflow) {                                              // lines shorter than assumed: more line slots
      if (ctx->min_line_bytes <= 1) return BVCF_E_TOO_LARGE;
      ctx->min_line_bytes /= 2;
      s->retries++;
      if (s->retries > 8) return BVCF_E_TOO_LARGE;
      const int rc = slot_enqueue(ctx, *s, false);
      if (rc) return rc;
      continue;
    }
    if (c.ev_overflow) {                                                // dense genotype block: more event slots
      ctx->ev_factor *= 4;
      s->retries++;
      if (s->retries > 8) return BVCF_E_TOO_LARGE;
      const int rc = slot_enqueue(ctx, *s, false);
      if (rc) return rc;
      continue;
    }
    if (c.row_overflow) { s->sc.row_cap = s->sc.row_cap * 4 + c.row_cursor; again = true; }  // MNP/multi-ALT heavy block
    if (c.out_overflow) {
      int rc = dev_reserve(ctx, s->d_out, (size_t)(c.out_cursor + c.out_cursor / 8 + 4096));
      if (rc) return rc;
      again = true;
    }
    if (dc.want_dosage && dc.n_samples > 0) {  // dosage rows, locus offsets and locus bytes grow to what the chunk reported
      if (c.row_cursor * (uint64_t)dc.n_samples > s->d_dosage.cap || c.row_cursor * 8 > s->d_loci_off.cap) {
        int rc = dev_reserve(ctx, s->d_dosage, (size_t)(c.row_cursor + 64) * dc.n_samples);
        if (rc) return rc;
        if ((rc = dev_reserve(ctx, s->d_loci_off, (size_t)(c.row_cursor + 64) * 8))) return rc;
        again = true;
      }
      if (c.loci_cursor > s->d_loci.cap) {
        int rc = dev_reserve(ctx, s->d_loci, (size_t)(c.loci_cursor + c.loci_cursor / 8 + 4096));
        if (rc) return rc;
        again = true;
      }
    }
    // every log line or none.  Compared with the capacity this chunk ran with: another slot may have raised ctx->diag_cap
    // since, and this slot's buffer is still the old size
    if (c.n_diags > s->diag_cap) { ctx->diag_cap = std::max(ctx->diag_cap, c.n_diags + c.n_diags / 4); again = true; }
    if (c.scratch_overflow) { s->sc.scratch_cap = c.scratch_cursor + c.scratch_cursor / 4 + (1ull << 20); again = true; }
    if (c.slow_overflow) { s->sc.slow_cap = c.n_slow + c.n_slow / 4 + 1024; again = true; }
    if (!again) break;
    s->retries++;
    if (s->retries > 8) return BVCF_E_TOO_LARGE;
    const int rc = slot_enqueue(ctx, *s, false);  // input is still on the device
    if (rc) return rc;
  }
  const RunCounters c = *s->h_ctr;
  // rows back to pinned host memory
  if (c.out_cursor > s->h_out_cap) {
    if (s->h_out) cudaFreeHost(s->h_out);
    s->h_out = nullptr;
    s->h_out_cap = 0;
    const size_t cap = (size_t)(c.out_cursor + c.out_cursor / 4 + 4096);
    CK(cudaMallocHost(&s->h_out, cap));
    s->h_out_cap = cap;
  }
  if (c.out_cursor) CK(cudaMemcpyAsync(s->h_out, s->d_out.p, c.out_cursor, cudaMemcpyDeviceToHost, s->stream));
  const bool dos = dc.want_dosage && dc.n_samples > 0;
  if (dos && c.row_cursor) {
    const size_t nb = (size_t)c.row_cursor * dc.n_samples;
    if (nb > s->h_dosage_cap) {
      if (s->h_dosage) cudaFreeHost(s->h_dosage);
      s->h_dosage = nullptr;
      CK(cudaMallocHost(&s->h_dosage, nb + nb / 4));
      s->h_dosage_cap = nb + nb / 4;
    }
    CK(cudaMemcpyAsync(s->h_dosage, s->d_dosage.p, nb, cudaMemcpyDeviceToHost, s->stream));
    if (c.loci_cursor > s->h_loci_cap) {
      if (s->h_loci) cudaFreeHost(s->h_loci);
      s->h_loci = nullptr; s->h_loci_cap = 0;
      const size_t cap = (size_t)(c.loci_cursor + c.loci_cursor / 4 + 4096);
      CK(cudaMallocHost(&s->h_loci, cap));
      s->h_loci_cap = cap;
    }
    if (c.row_cursor + 1 > s->h_loci_off_cap) {
      if (s->h_loci_off) cudaFreeHost(s->h_loci_off);
      s->h_loci_off = nullptr; s->h_loci_off_cap = 0;
      const size_t cap = (size_t)(c.row_cursor + c.row_cursor / 4 + 64);
      CK(cudaMallocHost(&s->h_loci_off, cap * 8));
      s->h_loci_off_cap = cap;
    }
    CK(cudaMemcpyAsync(s->h_loci, s->d_loci.p, c.loci_cursor, cudaMemcpyDeviceToHost, s->stream));
    CK(cudaMemcpyAsync(s->h_loci_off, s->d_loci_off.p, c.row_cursor * 8, cudaMemcpyDeviceToHost, s->stream));
  }
  // <= diag_cap: larger counts re-ran the chunk above.  A caller that takes no diagnostics does not pay for them: on
  // sites-only input with 9 % rejected alleles their copy, decode and sort was 3.6 ms of every 128 MiB chunk, more than
  // its PCIe time
  const uint32_t nd = (diags || n_diags) ? std::min(c.n_diags, s->diag_cap) : 0u;
  if (nd) {
    s->h_diag_raw.resize((size_t)nd * DIAG_WORDS);
    CK(cudaMemcpyAsync(s->h_diag_raw.data(), s->d_diags.p, (size_t)nd * DIAG_WORDS * 4, cudaMemcpyDeviceToHost, s->stream));
  }
  const auto t_kernels = std::chrono::steady_clock::now();
  CK(cudaStreamSynchronize(s->stream));
  const auto t_copied = std::chrono::steady_clock::now();
  if (tsv) *tsv = s->h_out;
  if (tsv_len) *tsv_len = (size_t)c.out_cursor;
  if (dosage) {
    memset(dosage, 0, sizeof(*dosage));
    dosage->n_samples = (uint32_t)dc.n_samples;
    if (dos && c.row_cursor) {
      s->h_loci_off[c.row_cursor] = c.loci_cursor;  // rows are packed in row order: row r ends where row r + 1 starts
      dosage->n_rows = c.row_cursor;
      dosage->dosage = s->h_dosage;
      dosage->loci = s->h_loci;
      dosage->loci_off = s->h_loci_off;
    }
  }
  decode_diags(s->h_diag_raw.data(), nd, s->h_diags);
  if (trace) {
    const auto t_end = std::chrono::steady_clock::now();
    auto ms = [](auto a, auto b) { return std::chrono::duration<double, std::milli>(b - a).count(); };
    fprintf(stderr, "[bvcf] collect %llu: wait %.2f ms, copy back %.2f ms (%llu B rows, %u diags), diags %.2f ms\n",
            (unsigned long long)seq, ms(t_begin, t_kernels), ms(t_kernels, t_copied), (unsigned long long)c.out_cursor, nd,
            ms(t_copied, t_end));
  }
  if (diags) *diags = s->h_diags.data();
  if (n_diags) *n_diags = s->h_diags.size();
  if (stats) {
    stats->n_lines = c.n_lines; stats->n_records = c.n_records; stats->n_rows = c.row_cursor;
    stats->in_bytes = s->len - s->skip; stats->out_bytes = c.out_cursor; stats->retries = s->retries;
  }
  return BVCF_OK;
}

int bvcf_release(bvcf_ctx *ctx, uint64_t seq) {
  if (!ctx) return BVCF_E_ARG;
  Slot *s = find_slot(ctx, seq);
  if (!s) return BVCF_E_STATE;
  s->busy = false;
  s->h_src = nullptr;
  return BVCF_OK;
}

// ---- resident path ----------------------------------------------------------------------------

int bvcf_resident_alloc(bvcf_ctx *ctx, size_t in_bytes, size_t out_capacity, void **d_in, void **d_out) {
  if (!ctx) return BVCF_E_ARG;
  cudaSetDevice(ctx->device);
  const uint64_t buf_len = round_up(in_bytes, 1024) + 2048;
  int rc;
  if ((rc = dev_reserve(ctx, ctx->r_in, buf_len + IN_SLACK))) return rc;
  if ((rc = dev_reserve(ctx, ctx->r_out, std::max<size_t>(out_capacity, 4096)))) return rc;
  CK(cudaMemset((uint8_t *)ctx->r_in.p + in_bytes, '\n', ctx->r_in.cap - in_bytes));
  ctx->r_in_bytes = in_bytes;
  if (d_in) *d_in = ctx->r_in.p;
  if (d_out) *d_out = ctx->r_out.p;
  return BVCF_OK;
}

int bvcf_resident_upload(bvcf_ctx *ctx, size_t offset, const void *host, size_t len) {
  if (!ctx || !host) return BVCF_E_ARG;
  if (offset + len > ctx->r_in_bytes) return BVCF_E_ARG;
  cudaSetDevice(ctx->device);
  CK(cudaMemcpy((uint8_t *)ctx->r_in.p + offset, host, len, cudaMemcpyHostToDevice));
  return BVCF_OK;
}

int bvcf_resident_run(bvcf_ctx *ctx, size_t len, bvcf_chunk_stats *stats, bvcf_kernel_times *times) {
  return bvcf_resident_run_at(ctx, 0, len, stats, times);
}

int bvcf_resident_run_at(bvcf_ctx *ctx, size_t begin, size_t len, bvcf_chunk_stats *stats, bvcf_kernel_times *times) {
  if (!ctx) return BVCF_E_ARG;
  if (!ctx->header_set) return BVCF_E_STATE;
  if (len > ctx->r_in_bytes || begin > len) return BVCF_E_ARG;
  cudaSetDevice(ctx->device);
  const DevCfg &dc = ctx->dcfg;
  uint32_t retries = 0;
  uint64_t launches0 = ctx->launches;
  std::vector<StageEvents> timing;
  for (;;) {
    int rc;
    if ((rc = scratch_reserve(ctx, ctx->r_sc, len - (begin & ~511ull), ctx->cfg.resident_subchunk_bytes))) return rc;
    if ((rc = dev_reserve(ctx, ctx->r_diags, (size_t)ctx->diag_cap * DIAG_WORDS * 4))) return rc;
    // the bytes after `len` must not look like data: pad (idempotent)
    const uint64_t buf_len = std::min<uint64_t>((ctx->r_in.cap - IN_SLACK) / 1024 * 1024, round_up(len, 1024) + 2048);
    CK(cudaMemsetAsync(ctx->r_d_ctr, 0, sizeof(RunCounters), ctx->r_stream));
    uint64_t dos_rows = 0;
    if (dc.want_dosage && dc.n_samples > 0)
      dos_rows = std::min<uint64_t>(ctx->r_dosage.cap / (uint64_t)dc.n_samples, ctx->r_loci_off.cap / 8);
    for (auto &t : timing)
      for (auto e : t.e) ctx->ev_pool.push_back(e);
    timing.clear();
    launches0 = ctx->launches;
    rc = enqueue_pipeline(ctx, ctx->r_sc, ctx->r_stream, (const uint8_t *)ctx->r_in.p, begin, len, buf_len,
                          (uint8_t *)ctx->r_out.p, ctx->r_out.cap, ctx->r_d_ctr, (int8_t *)ctx->r_dosage.p, dos_rows,
                          (uint8_t *)ctx->r_loci.p, ctx->r_loci.cap, (unsigned long long *)ctx->r_loci_off.p,
                          (uint32_t *)ctx->r_diags.p, ctx->diag_cap, times ? &timing : nullptr);
    if (rc) return rc;
    CK(cudaMemcpyAsync(ctx->r_h_ctr, ctx->r_d_ctr, sizeof(RunCounters), cudaMemcpyDeviceToHost, ctx->r_stream));
    CK(cudaStreamSynchronize(ctx->r_stream));
    const RunCounters &c = *ctx->r_h_ctr;
    bool again = false;
    if (c.slot_overflow) {  // lines shorter than assumed: more line slots, run again
      if (ctx->min_line_bytes <= 1) return BVCF_E_TOO_LARGE;
      ctx->min_line_bytes /= 2;
      if (++retries > 8) return BVCF_E_TOO_LARGE;
      continue;
    }
    if (c.ev_overflow) {  // dense genotype block: more event slots, run again
      ctx->ev_factor *= 4;
      if (++retries > 8) return BVCF_E_TOO_LARGE;
      continue;
    }
    if (c.row_overflow) { ctx->r_sc.row_cap = ctx->r_sc.row_cap * 4 + c.row_cursor; again = true; }
    if (c.scratch_overflow) { ctx->r_sc.scratch_cap = c.scratch_cursor + c.scratch_cursor / 4 + (1ull << 20); again = true; }
    if (c.n_diags > ctx->diag_cap) { ctx->diag_cap = c.n_diags + c.n_diags / 4; again = true; }
    if (c.slow_overflow) { ctx->r_sc.slow_cap = c.n_slow + c.n_slow / 4 + 1024; again = true; }
    if (c.out_overflow) {
      if ((rc = dev_reserve(ctx, ctx->r_out, (size_t)(c.out_cursor + c.out_cursor / 8 + 4096)))) return rc;
      again = true;
    }
    if (dc.want_dosage && dc.n_samples > 0) {
      if (c.row_cursor * (uint64_t)dc.n_samples > ctx->r_dosage.cap || c.row_cursor * 8 > ctx->r_loci_off.cap) {
        if ((rc = dev_reserve(ctx, ctx->r_dosage, (size_t)(c.row_cursor + 64) * dc.n_samples))) return rc;
        if ((rc = dev_reserve(ctx, ctx->r_loci_off, (size_t)(c.row_cursor + 64) * 8))) return rc;
        again = true;
      }
      if (c.loci_cursor > ctx->r_loci.cap) {
        if ((rc = dev_reserve(ctx, ctx->r_loci, (size_t)(c.loci_cursor + c.loci_cursor / 8 + 4096)))) return rc;
        again = true;
      }
    }
    if (!again) break;
    if (++retries > 8) return BVCF_E_TOO_LARGE;
  }
  const RunCounters &c = *ctx->r_h_ctr;
  ctx->r_last_records = c.n_records;
  ctx->r_last_len = len;
  if (stats) {
    stats->n_lines = c.n_lines; stats->n_records = c.n_records; stats->n_rows = c.row_cursor;
    stats->in_bytes = len - begin; stats->out_bytes = c.out_cursor; stats->retries = retries;
  }
  if (times) {
    memset(times, 0, sizeof(*times));
    for (auto &t : timing) {
      float ms;
      cudaEventElapsedTime(&ms, t.e[0], t.e[1]); times->scan_ms += ms;
      cudaEventElapsedTime(&ms, t.e[1], t.e[2]); times->compact_ms += ms;
      cudaEventElapsedTime(&ms, t.e[2], t.e[3]); times->stats_ms += ms;
      cudaEventElapsedTime(&ms, t.e[3], t.e[4]); times->rows_ms += ms;
      cudaEventElapsedTime(&ms, t.e[4], t.e[5]); times->names_ms += ms;
      cudaEventElapsedTime(&ms, t.e[3], t.e[6]); times->compose_ms += ms;
      cudaEventElapsedTime(&ms, t.e[7], t.e[4]); times->copyout_ms += ms;
    }
    if (!timing.empty()) cudaEventElapsedTime(&times->total_ms, timing.front().e[0], timing.back().e[5]);
    times->launches = (uint32_t)(ctx->launches - launches0);  // of the last (successful) attempt
    for (auto &t : timing)
      for (auto e : t.e) ctx->ev_pool.push_back(e);
  }
  return BVCF_OK;
}

// ---- bgzf input (SURVEY 8f-3) ------------------------------------------------------------------------------
// walk the gzip members of a bgzf buffer (RFC 1952 header with the "BC" extra subfield of the SAM spec 4.1).  The header
// rule is the one of bgzf.py block_size and bvcf_host.cpp bgzf_header: FLG has FEXTRA; the subfields of the extra field
// are walked in order, a subfield that runs past the end of the field ends the walk, and the first BC subfield with
// SLEN 2 gives BSIZE - 1.  Members with ISIZE 0 stay in the block table: the kernel checks that they inflate to nothing
// with CRC-32 0, so text hidden behind a zero ISIZE is refused instead of dropped.
static int bgzf_walk(const uint8_t *c, size_t n, std::vector<InflateBlock> *blocks, uint64_t *text_bytes) {
  size_t p = 0;
  uint64_t out = 0;
  while (p < n) {
    if (n - p < 18 || c[p] != 0x1f || c[p + 1] != 0x8b || c[p + 2] != 8 || !(c[p + 3] & 4)) return BVCF_E_ARG;
    const size_t xlen = (size_t)c[p + 10] | ((size_t)c[p + 11] << 8);
    if (n - p < 12 + xlen) return BVCF_E_ARG;
    size_t bsize = 0;
    for (size_t q = p + 12; q + 4 <= p + 12 + xlen;) {
      const size_t slen = (size_t)c[q + 2] | ((size_t)c[q + 3] << 8);
      if (q + 4 + slen > p + 12 + xlen) break;
      if (c[q] == 'B' && c[q + 1] == 'C' && slen == 2) { bsize = ((size_t)c[q + 4] | ((size_t)c[q + 5] << 8)) + 1; break; }
      q += 4 + slen;
    }
    if (bsize < 12 + xlen + 8 || n - p < bsize) return BVCF_E_ARG;  // not bgzf, or a truncated last block
    const uint32_t isize = (uint32_t)c[p + bsize - 4] | ((uint32_t)c[p + bsize - 3] << 8) | ((uint32_t)c[p + bsize - 2] << 16) |
                           ((uint32_t)c[p + bsize - 1] << 24);
    if (blocks) {
      InflateBlock b;
      b.in_off = p + 12 + xlen; b.in_len = (uint32_t)(bsize - 12 - xlen - 8); b.out_off = out; b.out_len = isize;
      b.crc = (uint32_t)c[p + bsize - 8] | ((uint32_t)c[p + bsize - 7] << 8) | ((uint32_t)c[p + bsize - 6] << 16) |
              ((uint32_t)c[p + bsize - 5] << 24);
      b.pad = 0;
      blocks->push_back(b);
    }
    out += isize;
    p += bsize;
  }
  if (text_bytes) *text_bytes = out;
  return BVCF_OK;
}

int bvcf_bgzf_text_bytes(const void *comp, size_t comp_len, uint64_t *text_bytes, uint64_t *n_blocks) {
  if (!comp || !text_bytes) return BVCF_E_ARG;
  std::vector<InflateBlock> blocks;
  const int rc = bgzf_walk((const uint8_t *)comp, comp_len, &blocks, text_bytes);
  if (n_blocks) *n_blocks = blocks.size();
  return rc;
}

int bvcf_resident_inflate_bgzf(bvcf_ctx *ctx, const void *comp, size_t comp_len, size_t dst_offset, size_t *text_bytes) {
  if (!ctx || !comp) return BVCF_E_ARG;
  cudaSetDevice(ctx->device);
  ctx->last_error.clear();
  std::vector<InflateBlock> blocks;
  uint64_t total = 0;
  int rc = bgzf_walk((const uint8_t *)comp, comp_len, &blocks, &total);
  if (rc) return rc;
  if (dst_offset + total > ctx->r_in_bytes) return BVCF_E_ARG;
  if (text_bytes) *text_bytes = (size_t)total;
  if (blocks.empty()) return BVCF_OK;
  if (blocks.size() >= (1ull << 32)) return BVCF_E_TOO_LARGE;
  for (auto &b : blocks) b.out_off += dst_offset;
  if ((rc = dev_reserve(ctx, ctx->r_comp, comp_len + 16))) return rc;
  if ((rc = dev_reserve(ctx, ctx->r_blocks, blocks.size() * sizeof(InflateBlock)))) return rc;
  if (!ctx->r_d_bad) CK(cudaMalloc(&ctx->r_d_bad, 4));
  CK(cudaMemcpyAsync(ctx->r_comp.p, comp, comp_len, cudaMemcpyHostToDevice, ctx->r_stream));  // the compressed bytes cross PCIe
  CK(cudaMemcpyAsync(ctx->r_blocks.p, blocks.data(), blocks.size() * sizeof(InflateBlock), cudaMemcpyHostToDevice, ctx->r_stream));
  CK(cudaMemsetAsync(ctx->r_d_bad, 0, 4, ctx->r_stream));
  InflateParams ip{};
  ip.comp = (const uint8_t *)ctx->r_comp.p; ip.out = (uint8_t *)ctx->r_in.p; ip.blocks = (const InflateBlock *)ctx->r_blocks.p;
  ip.n_blocks = (uint32_t)blocks.size(); ip.n_bad = ctx->r_d_bad;
  cudaFuncSetAttribute(bvcf_inflate_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)INF_SMEM);
  bvcf_inflate_kernel<<<ip.n_blocks, 32, INF_SMEM, ctx->r_stream>>>(ip);
  ctx->launches++;
  uint32_t bad = 0;
  CK(cudaMemcpyAsync(&bad, ctx->r_d_bad, 4, cudaMemcpyDeviceToHost, ctx->r_stream));
  CK(cudaStreamSynchronize(ctx->r_stream));
  if (bad) { ctx->last_error = std::to_string(bad) + " bgzf block(s) failed to inflate or failed their CRC-32 / ISIZE check"; return BVCF_E_ARG; }
  return BVCF_OK;
}

int bvcf_submit_bgzf(bvcf_ctx *ctx, uint64_t seq, const uint8_t *comp, size_t comp_len, size_t skip, const uint8_t *tail,
                     size_t tail_len) {
  if (!ctx || (!comp && comp_len) || (!tail && tail_len)) return BVCF_E_ARG;
  if (!ctx->header_set) return BVCF_E_STATE;
  if (find_slot(ctx, seq)) return BVCF_E_STATE;
  Slot *s = nullptr;
  for (auto &x : ctx->slots)
    if (!x.busy) { s = &x; break; }
  if (!s) return BVCF_E_STATE;
  ctx->last_error.clear();
  s->blocks.clear();
  uint64_t text = 0;
  int rc = comp_len ? bgzf_walk(comp, comp_len, &s->blocks, &text) : 0;
  if (rc) { ctx->last_error = "not whole bgzf blocks"; return rc; }
  if (skip > text) return BVCF_E_ARG;
  const uint64_t len = text + tail_len;
  if (len > ctx->cfg.max_chunk_bytes || len >= (1ull << 31) || s->blocks.size() >= (1ull << 31)) return BVCF_E_TOO_LARGE;
  if (tail_len && tail[tail_len - 1] != '\n') return BVCF_E_NOT_ALIGNED;  // (an empty tail: checked on the device)
  cudaSetDevice(ctx->device);
  // pinned staging: compressed bytes | block table | tail, so that the copies below are asynchronous
  const size_t tab_off = round_up(comp_len, 16), tail_off = tab_off + s->blocks.size() * sizeof(InflateBlock);
  const size_t need = tail_off + tail_len;
  if (need > s->h_stage_cap || !s->h_stage) {
    if (s->h_stage) cudaFreeHost(s->h_stage);
    s->h_stage = nullptr;
    s->h_stage_cap = 0;
    CK(cudaMallocHost(&s->h_stage, need + need / 4 + 4096));
    s->h_stage_cap = need + need / 4 + 4096;
  }
  if (comp_len) memcpy(s->h_stage, comp, comp_len);
  if (!s->blocks.empty()) memcpy(s->h_stage + tab_off, s->blocks.data(), s->blocks.size() * sizeof(InflateBlock));
  if (tail_len) memcpy(s->h_stage + tail_off, tail, tail_len);
  s->busy = true; s->seq = seq; s->h_src = nullptr; s->len = len; s->retries = 0;
  s->bgzf = true; s->skip = skip; s->text_len = text; s->tail_len = tail_len;
  rc = slot_enqueue(ctx, *s, true, comp_len);
  if (rc) s->busy = false;
  return rc;
}

int bvcf_diag_fields(bvcf_ctx *ctx, uint64_t seq, const uint8_t **text, const uint64_t **off) {
  if (!ctx || !text || !off) return BVCF_E_ARG;
  Slot *s = find_slot(ctx, seq);
  if (!s) return BVCF_E_STATE;
  cudaSetDevice(ctx->device);
  const size_t n = s->h_diags.size();
  s->h_field_off.assign(n + 1, 0);
  if (n) {
    if (n >= (1ull << 32)) return BVCF_E_TOO_LARGE;
    s->h_diag_starts.resize(n);
    for (size_t i = 0; i < n; i++) s->h_diag_starts[i] = s->h_diags[i].line_start;
    int rc;
    if ((rc = dev_reserve(ctx, s->d_diag_starts, n * 8))) return rc;
    if ((rc = dev_reserve(ctx, s->d_field_off, (n + 1) * 8))) return rc;
    CK(cudaMemcpyAsync(s->d_diag_starts.p, s->h_diag_starts.data(), n * 8, cudaMemcpyHostToDevice, s->stream));
    const unsigned long long *st = (const unsigned long long *)s->d_diag_starts.p;
    unsigned long long *fo = (unsigned long long *)s->d_field_off.p;
    bvcf_diag_fields_len_kernel<<<1, 1024, 0, s->stream>>>((const uint8_t *)s->d_in.p, s->len, st, (uint32_t)n, fo);
    ctx->launches++;
    CK(cudaMemcpyAsync(s->h_field_off.data(), fo, (n + 1) * 8, cudaMemcpyDeviceToHost, s->stream));
    CK(cudaStreamSynchronize(s->stream));
    const size_t total = (size_t)s->h_field_off[n];
    s->h_fields.resize(total);
    if (total) {
      if ((rc = dev_reserve(ctx, s->d_fields, total))) return rc;
      bvcf_diag_fields_copy_kernel<<<(unsigned)std::min<size_t>((n + 7) / 8, 1184), 256, 0, s->stream>>>(
          (const uint8_t *)s->d_in.p, st, fo, (uint32_t)n, (uint8_t *)s->d_fields.p);
      ctx->launches++;
      CK(cudaMemcpyAsync(s->h_fields.data(), s->d_fields.p, total, cudaMemcpyDeviceToHost, s->stream));
      CK(cudaStreamSynchronize(s->stream));
    }
    CK(cudaGetLastError());
  }
  *text = s->h_fields.data();
  *off = s->h_field_off.data();
  return BVCF_OK;
}

// ---- bgzf output (SURVEY 8f-4) -----------------------------------------------------------------------------
int bvcf_resident_download_bgzf(bvcf_ctx *ctx, size_t offset, size_t len, void *host, size_t host_cap, size_t *comp_len) {
  return bvcf_resident_download_bgzf_level(ctx, offset, len, 1, host, host_cap, comp_len);
}

int bvcf_resident_download_bgzf_level(bvcf_ctx *ctx, size_t offset, size_t len, int level, void *host, size_t host_cap,
                                      size_t *comp_len) {
  if (!ctx || !host || !comp_len || level < 1 || level > 9) return BVCF_E_ARG;
  if (offset + len > ctx->r_out.cap) return BVCF_E_ARG;
  *comp_len = 0;
  if (len == 0) return BVCF_OK;
  cudaSetDevice(ctx->device);
  const uint64_t nb64 = (len + DEF_SLICE - 1) / DEF_SLICE;
  if (nb64 >= (1ull << 31)) return BVCF_E_TOO_LARGE;
  const uint32_t nb = (uint32_t)nb64;
  int rc;
  if ((rc = dev_reserve(ctx, ctx->r_def_slots, (size_t)nb * DEF_SLOT))) return rc;
  if ((rc = dev_reserve(ctx, ctx->r_def_sizes, (size_t)nb * 4))) return rc;
  if ((rc = dev_reserve(ctx, ctx->r_def_offs, (size_t)nb * 8))) return rc;
  cudaStream_t st = ctx->r_stream;
  CK(cudaMemsetAsync(ctx->r_def_slots.p, 0, (size_t)nb * DEF_SLOT, st));  // the token bits are OR-ed in
  DeflateParams dp{};
  dp.text = (const uint8_t *)ctx->r_out.p + offset; dp.text_len = len; dp.slots = (uint8_t *)ctx->r_def_slots.p;
  dp.sizes = (uint32_t *)ctx->r_def_sizes.p; dp.n_blocks = nb;
  if (level == 1) bvcf_deflate_kernel<<<nb, 32, 0, st>>>(dp);
  else bvcf_deflate_dyn_kernel<<<nb, 32, def_dyn_smem(DEF_LEVELS[level]), st>>>(dp, DEF_LEVELS[level]);
  std::vector<uint32_t> sizes(nb);
  CK(cudaMemcpyAsync(sizes.data(), dp.sizes, (size_t)nb * 4, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  std::vector<unsigned long long> offs(nb);
  unsigned long long total = 0;
  for (uint32_t i = 0; i < nb; i++) {
    if (sizes[i] == 0) {  // bvcf_deflate_dyn_kernel's emitted bits disagree with its own count: a bug, never bad data
      ctx->last_error = "bgzf block " + std::to_string(i) + ": the deflate kernel's output disagrees with its size";
      return BVCF_E_CUDA;
    }
    offs[i] = total; total += sizes[i];
  }
  if (total > host_cap) { *comp_len = (size_t)total; return BVCF_E_TOO_LARGE; }  // comp_len says how much room it takes
  if ((rc = dev_reserve(ctx, ctx->r_def_out, (size_t)total + 16))) return rc;
  CK(cudaMemcpyAsync(ctx->r_def_offs.p, offs.data(), (size_t)nb * 8, cudaMemcpyHostToDevice, st));
  DeflatePackParams pp{};
  pp.slots = dp.slots; pp.sizes = dp.sizes; pp.offs = (const unsigned long long *)ctx->r_def_offs.p;
  pp.out = (uint8_t *)ctx->r_def_out.p; pp.n_blocks = nb;
  bvcf_deflate_pack_kernel<<<nb, 128, 0, st>>>(pp);
  ctx->launches += 2;
  CK(cudaMemcpyAsync(host, ctx->r_def_out.p, (size_t)total, cudaMemcpyDeviceToHost, st));  // the compressed rows cross PCIe
  CK(cudaStreamSynchronize(st));
  *comp_len = (size_t)total;
  return BVCF_OK;
}

int bvcf_resident_results(bvcf_ctx *ctx, bvcf_dosage_batch *dosage, const bvcf_diag **diags, size_t *n_diags) {
  if (!ctx) return BVCF_E_ARG;
  cudaSetDevice(ctx->device);
  const RunCounters &c = *ctx->r_h_ctr;
  const DevCfg &dc = ctx->dcfg;
  if (dosage) {
    memset(dosage, 0, sizeof(*dosage));
    dosage->n_samples = (uint32_t)dc.n_samples;
    if (dc.want_dosage && dc.n_samples > 0 && c.row_cursor) {
      ctx->r_h_dosage.resize((size_t)c.row_cursor * dc.n_samples);
      ctx->r_h_loci.resize((size_t)c.loci_cursor);
      ctx->r_h_loci_off.resize((size_t)c.row_cursor + 1);
      CK(cudaMemcpy(ctx->r_h_dosage.data(), ctx->r_dosage.p, ctx->r_h_dosage.size(), cudaMemcpyDeviceToHost));
      if (c.loci_cursor) CK(cudaMemcpy(ctx->r_h_loci.data(), ctx->r_loci.p, (size_t)c.loci_cursor, cudaMemcpyDeviceToHost));
      CK(cudaMemcpy(ctx->r_h_loci_off.data(), ctx->r_loci_off.p, (size_t)c.row_cursor * 8, cudaMemcpyDeviceToHost));
      ctx->r_h_loci_off[c.row_cursor] = c.loci_cursor;
      dosage->n_rows = c.row_cursor;
      dosage->dosage = ctx->r_h_dosage.data();
      dosage->loci = ctx->r_h_loci.data();
      dosage->loci_off = ctx->r_h_loci_off.data();
    }
  }
  ctx->r_h_diags.clear();
  const uint32_t nd = std::min<uint32_t>(c.n_diags, ctx->diag_cap);
  if (nd && ctx->r_diags.p) {
    std::vector<uint32_t> raw((size_t)nd * DIAG_WORDS);
    CK(cudaMemcpy(raw.data(), ctx->r_diags.p, raw.size() * 4, cudaMemcpyDeviceToHost));
    decode_diags(raw.data(), nd, ctx->r_h_diags);
  }
  if (diags) *diags = ctx->r_h_diags.data();
  if (n_diags) *n_diags = ctx->r_h_diags.size();
  return BVCF_OK;
}

int bvcf_resident_write_output(bvcf_ctx *ctx, size_t offset, const void *host, size_t len) {
  if (!ctx || !host) return BVCF_E_ARG;
  if (offset + len > ctx->r_out.cap) return BVCF_E_ARG;
  cudaSetDevice(ctx->device);
  CK(cudaMemcpy((uint8_t *)ctx->r_out.p + offset, host, len, cudaMemcpyHostToDevice));
  return BVCF_OK;
}

int bvcf_resident_download(bvcf_ctx *ctx, size_t offset, void *host, size_t len) {
  if (!ctx || !host) return BVCF_E_ARG;
  if (offset + len > ctx->r_out.cap) return BVCF_E_ARG;
  cudaSetDevice(ctx->device);
  CK(cudaMemcpy(host, (uint8_t *)ctx->r_out.p + offset, len, cudaMemcpyDeviceToHost));
  return BVCF_OK;
}

int bvcf_resident_peek(bvcf_ctx *ctx, size_t offset, void *host, size_t len) {
  if (!ctx || !host) return BVCF_E_ARG;
  if (offset + len > ctx->r_in.cap) return BVCF_E_ARG;
  cudaSetDevice(ctx->device);
  CK(cudaMemcpy(host, (uint8_t *)ctx->r_in.p + offset, len, cudaMemcpyDeviceToHost));
  return BVCF_OK;
}

int bvcf_resident_line_index(bvcf_ctx *ctx, uint64_t *starts, uint32_t *lens, uint32_t *an, size_t cap,
                             size_t *n_records) {
  if (!ctx) return BVCF_E_ARG;
  cudaSetDevice(ctx->device);
  // valid for single-sub-chunk runs: the dense table of the last sub-chunk
  const size_t n = (size_t)std::min<uint64_t>(ctx->r_h_ctr->chunk_records, cap);
  if (n_records) *n_records = ctx->r_h_ctr->chunk_records;
  if (n == 0) return BVCF_OK;
  std::vector<LineRec> tmp(n);
  CK(cudaMemcpy(tmp.data(), ctx->r_sc.dense.p, n * sizeof(LineRec), cudaMemcpyDeviceToHost));
  for (size_t i = 0; i < n; i++) {
    if (starts) starts[i] = tmp[i].start;
    if (lens) lens[i] = tmp[i].len;
    if (an) an[i] = tmp[i].an;
  }
  return BVCF_OK;
}

}  // extern "C"
