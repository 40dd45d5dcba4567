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
  float compact_ms;  /* line-table compaction + prefix sums */
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
