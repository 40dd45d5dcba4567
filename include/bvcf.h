/*
 * bvcf.h -- C ABI of libbvcf: the B200-native drop-in for bystro-vcf's per-line transform.
 *
 * The reference (Go, /root/reference/main.go) exposes no FFI; the seam this library sits behind is the
 * contract of processLines as driven by readVcf:
 *
 *   processLines(header []string, numChars int, config *Config, queue chan [][]byte,
 *                writer *bufio.Writer, complete chan bool, arrowWriter *ArrowWriter)     main.go:476-477
 *
 * i.e. "given the parsed #CHROM header, the EOL width and the Config, turn batches of complete
 * newline-terminated data lines into TSV rows (+ dosage rows)".  Each entry point below cites the
 * reference lines it replaces.  INTEGRATION.md shows the cgo binding a maintainer would add.
 *
 * Conventions: plain C types only; one bvcf_ctx per GPU, used by one host thread at a time; no global
 * state; every function returns 0 on success or a negative BVCF_E_* code (never abort()/exit()).
 * There is no CPU fallback: without a usable CUDA device bvcf_create fails with BVCF_E_CUDA.
 */
#ifndef BVCF_H
#define BVCF_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BVCF_ABI_VERSION 2

typedef struct bvcf_ctx bvcf_ctx;

/* Mirrors the Config fields processLines reads (main.go:494-503) + numChars (main.go:250). */
typedef struct {
  const char *empty_field;     /* --emptyField      main.go:91   default "!"  (any byte string <= 63 B) */
  const char *field_delim;     /* --fieldDelimiter  main.go:92   default ";"  (any byte string <= 63 B) */
  int keep_id;                 /* --keepId          main.go:93,679 */
  int keep_info;               /* --keepInfo        main.go:96,684 */
  int keep_pos;                /* --keepPos         main.go:95,674 */
  int want_tsv;                /* !--noOut          main.go:502 (needsLabels) */
  int want_dosage;             /* --dosageOutput set  main.go:503 (needsDosages) */
  const char *const *allow;    /* --allowFilter, already split+trimmed  main.go:108-114 */
  int n_allow;                 /* < 0 => nil map => every FILTER value allowed ("" or "*") */
  const char *const *exclude;  /* --excludeFilter   main.go:117-123 */
  int n_exclude;               /* 0 => nil map */
  int eol_width;               /* numChars: 1 "\n", 2 "\r\n"   main.go:250,535 */
  int normalize_dots;          /* parse.NormalizeHeader: '.' -> '_' in sample names  main.go:296 */
  /* tuning; 0 = library default */
  int n_slots;                 /* host chunks in flight (streams), default 3 */
  size_t max_chunk_bytes;      /* largest host chunk bvcf_submit will be given, default 256 MiB */
  size_t resident_subchunk_bytes; /* device-resident runs are cut into equal pieces of at most this size, default 24 GiB */
} bvcf_config;

/* error codes */
enum {
  BVCF_OK = 0,
  BVCF_E_ARG = -1,        /* bad argument / config */
  BVCF_E_CUDA = -2,       /* CUDA runtime error (no device, OOM, launch failure); see bvcf_last_error */
  BVCF_E_STATE = -3,      /* call order (no header set, unknown seq, slot busy) */
  BVCF_E_NOT_ALIGNED = -4,/* chunk does not end with '\n' */
  BVCF_E_TOO_LARGE = -5,  /* chunk > max_chunk_bytes, > 2^20 samples, header too wide ... */
  BVCF_E_NOMEM = -6
};

/* diagnostics: what the reference logs with log.Printf and then skips (main.go:41-51,730-986) */
enum {
  BVCF_DIAG_SAME = 1,    /* "REF == ALT"            "%s:%s : %s"        main.go:730 */
  BVCF_DIAG_BAD_ALT = 2, /* "ALT not ACTG"          "%s:%s ALT #%d %s"  main.go:737,782 */
  BVCF_DIAG_DEL1 = 3,    /* "1st base REF != ALT"   "%s:%s ALT #1 %s"   main.go:748 */
  BVCF_DIAG_POS = 4,     /* "Invalid POS"           "%s:%s ALT #1 %s"   main.go:755 */
  BVCF_DIAG_INS1 = 5,    /* "1st base ALT != REF"   "%s:%s ALT #%d %s"  main.go:798 */
  BVCF_DIAG_MIXED = 6,   /* "Mixed indel/snp sites not supported"   "%s:%s ALT#%d %s"  main.go:934,986 */
  BVCF_DIAG_DEL1_LIST = 7, /* DEL1 inside the ALT list: "%s:%s ALT#%d %s" (no space)  main.go:835 */
  BVCF_DIAG_POS_LIST = 8   /* POS inside the ALT list:  "%s:%s %s"                    main.go:827 */
};
typedef struct {
  uint64_t line_no;    /* 0-based data-line index within the chunk */
  int32_t alt_no;      /* 1-based ALT number; 0 if the message carries none */
  int32_t code;        /* BVCF_DIAG_* */
  uint64_t line_start; /* byte offset of that line in the chunk (its CHROM and POS fields start the log text) */
} bvcf_diag;

/* One chunk's share of the dosage matrix (main.go:576-584): row i is locus i + n_samples int8. */
typedef struct {
  uint64_t n_rows;
  uint32_t n_samples;
  const int8_t *dosage;      /* n_rows x n_samples, row-major (pinned host memory) */
  const uint8_t *loci;       /* concatenated "chrom:pos:ref:alt" strings */
  const uint64_t *loci_off;  /* n_rows + 1 offsets into loci */
} bvcf_dosage_batch;

typedef struct {
  uint64_t n_lines;   /* newline-terminated data lines seen */
  uint64_t n_records; /* lines with the header's field count (main.go:449) */
  uint64_t n_rows;    /* TSV rows emitted */
  uint64_t in_bytes;
  uint64_t out_bytes;
  uint32_t retries;   /* scratch-capacity retries (dense genotype blocks) */
} bvcf_chunk_stats;

/* per-kernel device time of the last resident run, CUDA events on the launching stream */
typedef struct {
  float scan_ms;     /* bvcf_scan_genotype_kernel: newline/tab index + per-sample GT classify  (north-star kernels 1+3) */
  float compact_ms;  /* line-table compaction + prefix sums (+ the region filter, with regions set) */
  float stats_ms;    /* bvcf_line_stats_kernel: het/hom/missing/ac/an per record (kernel 3, reduction half) */
  float rows_ms;     /* bvcf_tile_kernel: FILTER + getAlleles + row text, offsets by decoupled look-back, rows and short
                        sample-name lists written in one pass (kernels 2+4) */
  float names_ms;    /* bvcf_names_{vec,long,big}_kernel: long sample-name lists + their dosage rows (kernel 4b) */
  float total_ms;    /* first launch to last launch, whole run */
  uint32_t launches; /* kernels launched */
  float compose_ms;  /* inside rows_ms: bvcf_compose_kernel */
  float copyout_ms;  /* inside rows_ms: the copy-out and slow-path kernels (the rest of rows_ms is the tile-offset scan) */
} bvcf_kernel_times;

/* ---- lifecycle --------------------------------------------------------------------------- */

/* Replaces Config capture at main.go:494-503.  Copies everything it needs from cfg. */
int bvcf_create(bvcf_ctx **out, int cuda_device, const bvcf_config *cfg);
void bvcf_destroy(bvcf_ctx *ctx);

/* TSV header line without trailing newline (stringHeader, main.go:219-239).
 * Returns the length; writes at most cap bytes (NUL-terminated when it fits). */
int bvcf_header_line(const bvcf_config *cfg, char *buf, size_t cap);

/* The "#CHROM\tPOS..." line, with or without its EOL (main.go:281-296,505-509): fixes the required
 * field count and uploads the (normalised) sample-name table. */
int bvcf_set_header(bvcf_ctx *ctx, const char *chrom_line, size_t len);

/* Regions (--regions / --regionsFile): only the records inside them are transformed, by both the streaming slots and the
 * resident path.  Region i is contig chrom[i] (matched byte for byte against CHROM) and the 1-based inclusive positions
 * [beg[i], end[i]]: a record is kept when its POS is 1 to 18 ASCII digits whose value lies in a region of its CHROM --
 * bcftools view -t (targets) semantics: a deletion that starts before a region and reaches into it is not kept.  Other
 * records give no row, no dosage row and no diagnostic, as if their lines were not in the input; line numbers and
 * bvcf_chunk_stats' n_lines / n_records still count them.  The regions are copied (overlapping and adjacent ones
 * merged); n == 0 clears them.  BVCF_E_ARG: a NULL or empty name, beg < 1 or beg > end.  BVCF_E_STATE: a chunk is in
 * flight. */
int bvcf_set_regions(bvcf_ctx *ctx, const char *const *chrom, const int64_t *beg, const int64_t *end, size_t n);

/* Host only: the bgzf virtual-offset spans [spans[2k], spans[2k + 1]) that hold every record of the regions (given as to
 * bvcf_set_regions) a tabix or CSI index knows of.  `index` is the index file after gzip decompression ("TBI\1" or
 * "CSI\1"); the spans are sorted and disjoint, start and end at record boundaries, and may hold records outside the
 * regions too (bvcf_set_regions drops those).  A contig the index does not list gives no span.  *n_spans receives the
 * count; BVCF_E_TOO_LARGE when it is more than cap, BVCF_E_ARG on a malformed index or region. */
int bvcf_index_spans(const void *index, size_t len, const char *const *chrom, const int64_t *beg, const int64_t *end,
                     size_t n, uint64_t *spans, size_t cap, size_t *n_spans);

/* ---- streaming path: host chunks in, host rows out (the workQueue contract, main.go:353-380) ---- */

/* Pinned host memory so that submit's H2D copy and collect's D2H copy are truly asynchronous. */
int bvcf_host_alloc(void **ptr, size_t bytes);
void bvcf_host_free(void *ptr);

/* Enqueue one newline-aligned chunk of data lines (H2D + all kernels) on a free slot's stream and
 * return immediately.  The caller keeps ownership of `chunk` and must keep it alive until
 * bvcf_collect(seq) returns.  BVCF_E_STATE if n_slots chunks are already in flight. */
int bvcf_submit(bvcf_ctx *ctx, uint64_t seq, const uint8_t *chunk, size_t len);

/* Wait for chunk `seq`; rows are in input order.  tsv / dosage / diags point into library-owned
 * pinned memory valid until bvcf_release(seq).  dosage, diags, stats may be NULL. */
int bvcf_collect(bvcf_ctx *ctx, uint64_t seq, const uint8_t **tsv, size_t *tsv_len,
                 bvcf_dosage_batch *dosage, const bvcf_diag **diags, size_t *n_diags,
                 bvcf_chunk_stats *stats);
int bvcf_release(bvcf_ctx *ctx, uint64_t seq);

/* A chunk given as whole bgzf blocks: its text is inflate(comp)[skip:] followed by tail[0..tail_len), and must end
 * with '\n'.  The CRC-32 and ISIZE of every member are checked on the device; bvcf_collect(seq) returns BVCF_E_ARG on
 * a corrupt member.  The caller keeps comp and tail alive until bvcf_collect(seq) returns.  max_chunk_bytes limits the
 * inflated text plus the tail; a diagnostic's line_start is an offset into inflate(comp) followed by the tail. */
int bvcf_submit_bgzf(bvcf_ctx *ctx, uint64_t seq, const uint8_t *comp, size_t comp_len, size_t skip,
                     const uint8_t *tail, size_t tail_len);
/* CHROM and POS ("CHROM<TAB>POS", back to back) of the line of each diagnostic of collected chunk seq, in the order
 * bvcf_collect returned them; off has n_diags + 1 entries.  Gathered on the device: the text of a bgzf chunk exists
 * only there.  Library-owned, valid until bvcf_release(seq). */
int bvcf_diag_fields(bvcf_ctx *ctx, uint64_t seq, const uint8_t **text, const uint64_t **off);

/* ---- device-resident path: input already in HBM (bench `value`, torch/cupy interop) -------- */

/* (Re)allocate the context's resident input region (+ padding) and output region; returns device pointers. */
int bvcf_resident_alloc(bvcf_ctx *ctx, size_t in_bytes, size_t out_capacity, void **d_in, void **d_out);
/* Convenience H2D into the resident input region. */
int bvcf_resident_upload(bvcf_ctx *ctx, size_t offset, const void *host, size_t len);
/* Run the whole pipeline over data lines in [0, len) of the resident region (must end with '\n').
 * No host<->device traffic except a few counters at the end. */
int bvcf_resident_run(bvcf_ctx *ctx, size_t len, bvcf_chunk_stats *stats, bvcf_kernel_times *times);
/* The same over data lines in [begin, len): what comes before `begin` (meta lines, the #CHROM line of a file that was
 * inflated whole) is not looked at.  `begin` must be the first byte of a line. */
int bvcf_resident_run_at(bvcf_ctx *ctx, size_t begin, size_t len, bvcf_chunk_stats *stats, bvcf_kernel_times *times);

/* bgzf-compressed input (bgzip / htslib .vcf.gz; upstream of main.go:192 the reference pipes through `pigz -d -c`,
 * README.md:10,46): only the COMPRESSED bytes cross PCIe, the DEFLATE blocks are inflated on the GPU (one warp per
 * bgzf block, its CRC-32 and ISIZE checked) straight into the resident input region at `dst_offset`.  `comp` must hold
 * whole bgzf blocks.  text_bytes receives the uncompressed size.  BVCF_E_ARG: not bgzf, corrupt (including a CRC-32
 * mismatch), or larger than the region. */
int bvcf_resident_inflate_bgzf(bvcf_ctx *ctx, const void *comp, size_t comp_len, size_t dst_offset, size_t *text_bytes);
/* Host only: the uncompressed size (sum of ISIZE) and block count of a bgzf buffer of whole blocks.  Every member is
 * counted, those with ISIZE 0 (the EOF block among them) too: the GPU inflates and checks them like any other. */
int bvcf_bgzf_text_bytes(const void *comp, size_t comp_len, uint64_t *text_bytes, uint64_t *n_blocks);

/* ---- bgzf input on the host: what a host needs to read a .vcf.gz before its groups go to the GPU ---- */

/* Host only: the bgzf block at p[0, n) -- a gzip member with FLG.FEXTRA whose extra field holds a BC subfield with
 * SLEN 2 anywhere in it (SAM spec 4.1; the first such subfield gives BSIZE - 1).  *size receives 0 while the header is
 * not complete in n bytes, else BSIZE -- also when the block is then refused as corrupt, so *size > 0 tells a bgzf
 * header.  When the whole block is in p[0, n), *isize receives its ISIZE, and a block with ISIZE 0 is inflated and
 * refused unless it holds no text.  BVCF_E_ARG with a static reason in *why: not a bgzf block, no BC subfield, smaller
 * than its header and trailer, or corrupt. */
int bvcf_bgzf_block(const void *p, size_t n, size_t *size, uint32_t *isize, const char **why);
/* Host only: bvcf_bgzf_block over the blocks that follow each other from p on: the first cap of them, or those before
 * the first that is not whole in p[0, n), give size[k] and isize[k]; *n_blocks receives their count (on a refusal, the
 * count of those before the refused one). */
int bvcf_bgzf_blocks(const void *p, size_t n, uint32_t *size, uint32_t *isize, size_t cap, size_t *n_blocks,
                     const char **why);
/* Host only: inflate the whole bgzf block at block[0, n) into text[0, ISIZE) with zlib and check its CRC-32 and ISIZE.
 * BVCF_E_ARG with a static reason in *why: not bgzf, truncated or corrupt; BVCF_E_TOO_LARGE: cap < ISIZE. */
int bvcf_bgzf_inflate(const void *block, size_t n, void *text, size_t cap, const char **why);

/* Block i of the input for bvcf_bgzf_plan: a block with text (those with ISIZE 0 already checked and left out). */
typedef struct {
  const uint8_t *bytes; /* its first byte: read only before the next call of the block function */
  size_t size;          /* BSIZE */
  uint64_t start;       /* text offset of its first byte: the sum of the ISIZEs before it */
  uint32_t isize;
} bvcf_bgzf_blk;
/* 1 with *b filled, 0 past the last block, < 0 an error that ends the plan */
typedef int (*bvcf_bgzf_block_fn)(void *user, size_t i, bvcf_bgzf_blk *b);
/* one group, blocks [lo_block, hi_block): its text is inflate(blocks)[skip:] + tail; non-zero ends the plan */
typedef int (*bvcf_bgzf_emit_fn)(void *user, size_t lo_block, size_t hi_block, size_t skip, const uint8_t *tail,
                                 size_t tail_len);
/* Host only: cut an input into the groups of whole blocks that bvcf_submit_bgzf takes, data lines from text offset
 * data_off (the end of the #CHROM line) on, and hand each group to emit in input order.
 *  - A group's blocks are taken while its text is below chunk_bytes; the first group starts at the block holding text
 *    byte data_off, its skip is where data_off falls in it.
 *  - The line that crosses into the next group belongs to this one: its continuation -- the next group's text up to and
 *    including its first newline, inflated here -- is this group's tail and the next group's skip.  A next group with
 *    no newline joins this one.
 *  - The last group ends at the input's last newline (an unterminated last line is dropped): the blocks from the one
 *    holding it on are inflated here and left out, their text up to it is the tail.  What is left of the data inside the
 *    block of that newline goes to the tail of the group before.
 *  - A group whose text plus tail exceeds cap is refused: BVCF_E_TOO_LARGE, *why "a single line exceeds the chunk
 *    capacity; raise --chunkBytes".
 * Blocks are asked for in order, i = 0, 1, 2, ... until block returns 0, and block i once more right before its bytes are
 * read.  Once emit returns for a group, the planner reads no block bytes before that group's hi_block, so a reader may
 * drop them.  A non-zero return of a callback ends the plan and is returned; a corrupt block inflated here gives
 * BVCF_E_ARG and its reason in *why. */
int bvcf_bgzf_plan(bvcf_bgzf_block_fn block, bvcf_bgzf_emit_fn emit, void *user, uint64_t data_off, size_t chunk_bytes,
                   size_t cap, const char **why);

/* bgzf-compressed output (downstream of the reference stands `| pigz -c`, README.md:10,71): the rows in
 * [offset, offset + len) of the resident output region are deflated on the GPU (48 KiB slices, LZ77 + fixed Huffman
 * codes, CRC-32) and only the compressed blocks cross PCIe.  The bytes are whole bgzf blocks: concatenate the
 * pieces of a file and end it with the 28-byte bgzf EOF block.  BVCF_E_TOO_LARGE: host_cap is too small, *comp_len
 * says what is needed. */
int bvcf_resident_download_bgzf(bvcf_ctx *ctx, size_t offset, size_t len, void *host, size_t host_cap, size_t *comp_len);
/* The same at a compression level, as `bgzip -l` / `pigz -N` take one: 1 is bvcf_resident_download_bgzf (the bytes are
 * the same); 2..9 search more match candidates per position (from 4 on, lazily) and pick per block the cheapest of
 * dynamic Huffman codes, fixed codes and a stored block.  Any other level: BVCF_E_ARG. */
int bvcf_resident_download_bgzf_level(bvcf_ctx *ctx, size_t offset, size_t len, int level, void *host, size_t host_cap,
                                      size_t *comp_len);

/* Put host bytes into the resident output region (a host that wants its own text -- the TSV header line, say --
 * to leave through bvcf_resident_download_bgzf with the rows). */
int bvcf_resident_write_output(bvcf_ctx *ctx, size_t offset, const void *host, size_t len);

/* What the last bvcf_resident_run[_at] produced besides the rows: the dosage batch (when the context was created
 * with want_dosage) and the diagnostics; line_start offsets are into the resident input region.  Library-owned
 * memory, valid until the next resident run.  Either pointer may be NULL. */
int bvcf_resident_results(bvcf_ctx *ctx, bvcf_dosage_batch *dosage, const bvcf_diag **diags, size_t *n_diags);

/* Copy `len` output bytes starting at `offset` back to the host. */
int bvcf_resident_download(bvcf_ctx *ctx, size_t offset, void *host, size_t len);
/* Copy `len` bytes of the resident INPUT region back to the host (device-generated workloads). */
int bvcf_resident_peek(bvcf_ctx *ctx, size_t offset, void *host, size_t len);

/* ---- introspection ----------------------------------------------------------------------- */

/* Line index of the last resident run (north-star kernel 1's product): copies up to cap entries.
 * starts[i] = byte offset of record i, lens[i] = its length incl. EOL, an[i] = non-missing allele count. */
int bvcf_resident_line_index(bvcf_ctx *ctx, uint64_t *starts, uint32_t *lens, uint32_t *an, size_t cap,
                             size_t *n_records);

const char *bvcf_strerror(int rc);
const char *bvcf_last_error(const bvcf_ctx *ctx); /* detail of the last BVCF_E_CUDA */
int bvcf_abi_version(void);
/* number of kernel launches this context has made so far */
uint64_t bvcf_launch_count(const bvcf_ctx *ctx);

#ifdef __cplusplus
}
#endif
#endif /* BVCF_H */
