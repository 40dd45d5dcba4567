// bvcf_host.cpp -- `bystro-vcf-b200`: the reference's main()/readVcf (main.go:134-396) as a C++ host over the
// libbvcf C ABI.  Same flags, same stdin/stdout contract, so it drops into
//     pigz -d -c in.vcf.gz | bystro-vcf-b200 --keepId --keepInfo | pigz -c > out.gz
// The per-line work happens on the GPU(s).  Threads mirror the reference's producer + worker pool
// (main.go:345-380) with GPUs as the workers:
//   reader     finds newline-aligned chunk boundaries; stdin is read straight into pinned buffers, a regular
//              --in file is memory-mapped and only the boundaries are computed here.  A .vcf.gz (bgzf) input is cut
//              into groups of whole blocks instead (BgzfIn, bvcf_bgzf_plan): the compressed bytes go to the GPUs;
//   GPU worker one per GPU (chunk k goes to GPU k mod N): stages its chunks into its own pinned ring (parallel
//              memcpy out of the mapping), keeps n_slots chunks in flight on its context, and -- when it is chunk
//              k's turn -- writes the rows, appends the dosage batch to the Arrow file and logs the diagnostics,
//              so everything leaves in input order while the other GPUs keep working.
// (The reference is Go; no Go toolchain exists in this image, so the host is C++ -- see INTEGRATION.md for
// the equivalent cgo binding.)
#include <cerrno>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <algorithm>
#include <condition_variable>
#include <deque>
#include <mutex>
#include <memory>
#include <string>
#include <thread>
#include <vector>

#include <fcntl.h>
#include <zlib.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

#include "../../include/bvcf.h"
#ifndef BVCF_NO_ARROW
#include "bvcf_arrow.h"
#endif

namespace {

struct Config {  // main.go:63-80
  std::string inPath, outPath, dosageMatrixOutPath, sampleListPath, famPath, errPath, cpuProfile;
  std::string emptyField = "!", fieldDelimiter = ";";
  bool noOut = false, keepID = false, keepInfo = false, keepQual = false, keepPos = false;
  bool allowAll = false;  // allowedFilters == nil
  std::vector<std::string> allowed, excluded;
  // not in the reference
  int gpus = 1;
  std::vector<int> devices;  // --devices a,b,...: CUDA device of each worker (a device may be listed twice); default 0..gpus-1
  size_t chunkBytes = 64u << 20;
  bool bgzfOut = false;  // --bgzfOut: the rows leave as bgzf blocks deflated on the GPU (the `| pigz -c` of README.md:10,71)
  int bgzfLevel = 1;     // --bgzfLevel N: 1..9 as `bgzip -l` / `pigz -N` take it (bvcf_resident_download_bgzf_level)
  // --regions / --regionsFile: only the records inside these (contig, 1-based inclusive [beg, end]) are transformed
  bool regionsSet = false;
  std::vector<std::string> regionChrom;
  std::vector<int64_t> regionBeg, regionEnd;
};

std::string trim(const std::string &s) {  // strings.TrimSpace
  size_t a = 0, b = s.size();
  while (a < b && isspace((unsigned char)s[a])) a++;
  while (b > a && isspace((unsigned char)s[b - 1])) b--;
  return s.substr(a, b - a);
}
std::vector<std::string> split_trim(const std::string &s) {
  std::vector<std::string> out;
  size_t p = 0;
  for (;;) {
    size_t q = s.find(',', p);
    out.push_back(trim(s.substr(p, q == std::string::npos ? std::string::npos : q - p)));
    if (q == std::string::npos) break;
    p = q + 1;
  }
  return out;
}

// The reader thread and the GPU workers may fail at once: the first message wins, and the process ends without running
// exit-time teardown (the CUDA runtime's among it) under threads that are still inside CUDA calls.  Output goes
// through write(2), so nothing is left in a stdio buffer.
[[noreturn]] void fatal(const std::string &msg) {  // log.Fatal
  static std::mutex m;
  m.lock();
  fprintf(stderr, "%s\n", msg.c_str());
  fflush(stderr);
  _exit(1);
}

// strconv.ParseInt(s, 0, 64), what Go's `flag` package reads an int flag with: a sign, then 0x / 0o / 0b / 0 (octal)
// prefixes or decimal digits, underscores between digits
bool go_int(const std::string &s, long long *out) {
  size_t i = 0;
  const bool neg = !s.empty() && s[0] == '-';
  if (!s.empty() && (s[0] == '-' || s[0] == '+')) i = 1;
  int base = 10;
  if (s.size() > i + 1 && s[i] == '0') {
    const char b = (char)tolower((unsigned char)s[i + 1]);
    if (b == 'x') base = 16, i += 2;
    else if (b == 'o') base = 8, i += 2;
    else if (b == 'b') base = 2, i += 2;
    else base = 8, i += 1;
  }
  if (i >= s.size()) return false;
  unsigned long long v = 0;
  bool digit_before = base == 8 && s[i - 1] == '0';  // "0_7" is octal 7
  for (; i < s.size(); i++) {
    if (s[i] == '_') {
      if (!digit_before || i + 1 >= s.size() || s[i + 1] == '_') return false;
      continue;
    }
    const int c = tolower((unsigned char)s[i]);
    const int d = isdigit(c) ? c - '0' : (c >= 'a' && c <= 'z') ? c - 'a' + 10 : 99;
    if (d >= base) return false;
    if (v > (~0ull - (unsigned)d) / (unsigned)base) return false;
    v = v * (unsigned)base + (unsigned)d;
    digit_before = true;
  }
  if (v > (neg ? (1ull << 63) : (1ull << 63) - 1)) return false;
  *out = neg ? (long long)(0 - v) : (long long)v;
  return true;
}

// a decimal number of 0..2^63-1 (no sign): what --regions and --regionsFile positions are
bool pos_int(const std::string &s, int64_t *out) {
  if (s.empty() || s.size() > 19) return false;
  unsigned long long v = 0;
  for (char ch : s) {
    if (ch < '0' || ch > '9') return false;
    v = v * 10 + (unsigned)(ch - '0');
  }
  if (v > (unsigned long long)INT64_MAX) return false;
  *out = (int64_t)v;
  return true;
}

// --regions chr|chr:pos|chr:beg-end|chr:beg-[,...] (bcftools -r): the position part follows the last ':'
void parse_regions(const std::string &arg, Config &c) {
  size_t p = 0;
  for (;;) {
    const size_t q = arg.find(',', p);
    const std::string item = arg.substr(p, q == std::string::npos ? std::string::npos : q - p);
    auto bad = [&]() { fatal("--regions: malformed region \"" + item + "\""); };
    if (item.empty()) bad();
    const size_t colon = item.rfind(':');
    std::string chrom = item;
    int64_t beg = 1, end = INT64_MAX;
    if (colon != std::string::npos) {
      chrom = item.substr(0, colon);
      const std::string r = item.substr(colon + 1);
      const size_t dash = r.find('-');
      if (dash == std::string::npos) {
        if (!pos_int(r, &beg)) bad();
        end = beg;
      } else {
        if (!pos_int(r.substr(0, dash), &beg)) bad();
        if (dash + 1 < r.size() && !pos_int(r.substr(dash + 1), &end)) bad();
      }
      if (beg < 1 || beg > end) bad();
    }
    if (chrom.empty()) bad();
    c.regionChrom.push_back(chrom); c.regionBeg.push_back(beg); c.regionEnd.push_back(end);
    if (q == std::string::npos) break;
    p = q + 1;
  }
}

// --regionsFile: BED (0-based, half-open): "#", "track" and "browser" lines and blank lines are skipped, columns past the
// third are ignored; an empty interval holds no position
void parse_regions_file(const std::string &path, Config &c) {
  FILE *f = fopen(path.c_str(), "r");
  if (!f) fatal("--regionsFile: " + path + ": " + strerror(errno));
  std::string line;
  size_t line_no = 0;
  for (int ch = 0; ch != EOF;) {
    line.clear();
    while ((ch = fgetc(f)) != EOF && ch != '\n') line += (char)ch;
    line_no++;
    if (!line.empty() && line.back() == '\r') line.pop_back();
    std::vector<std::string> col;
    for (size_t i = 0; i < line.size();) {
      while (i < line.size() && (line[i] == '\t' || line[i] == ' ')) i++;
      size_t j = i;
      while (j < line.size() && line[j] != '\t' && line[j] != ' ') j++;
      if (j > i) col.push_back(line.substr(i, j - i));
      i = j;
    }
    if (col.empty() || col[0][0] == '#' || col[0] == "track" || col[0] == "browser") continue;
    int64_t b, e;
    const std::string where = "--regionsFile: " + path + " line " + std::to_string(line_no) + ": ";
    if (col.size() < 3) { fclose(f); fatal(where + "fewer than three columns"); }
    if (!pos_int(col[1], &b) || !pos_int(col[2], &e)) { fclose(f); fatal(where + "start and end must be non-negative integers"); }
    if (b > e) { fclose(f); fatal(where + "start > end"); }
    if (b == e) continue;
    c.regionChrom.push_back(col[0]); c.regionBeg.push_back(b + 1); c.regionEnd.push_back(e);
  }
  fclose(f);
}

// Go `flag` syntax: -x / --x, --x=v / --x v; bool flags --x or --x=true|false; stops at the first non-flag.
Config setup(int argc, char **argv) {  // main.go:82-126
  Config c;
  std::string allow = "PASS,.", exclude;
  struct SF { const char *name; std::string *dst; };
  const SF sf[] = {{"in", &c.inPath}, {"fam", &c.famPath}, {"err", &c.errPath}, {"out", &c.outPath},
                   {"dosageOutput", &c.dosageMatrixOutPath}, {"sample", &c.sampleListPath},
                   {"emptyField", &c.emptyField}, {"fieldDelimiter", &c.fieldDelimiter}, {"cpuProfile", &c.cpuProfile},
                   {"allowFilter", &allow}, {"excludeFilter", &exclude}};
  struct BF { const char *name; bool *dst; };
  const BF bf[] = {{"noOut", &c.noOut}, {"keepId", &c.keepID}, {"keepQual", &c.keepQual}, {"keepPos", &c.keepPos},
                   {"keepInfo", &c.keepInfo}, {"bgzfOut", &c.bgzfOut}};
  std::string gpus, chunk, devices, level;
  bool level_given = false;
  std::vector<std::pair<bool, std::string>> regions;  // (is a file, value) in flag order
  for (int i = 1; i < argc; i++) {
    std::string s = argv[i];
    if (s.size() < 2 || s[0] != '-') break;
    if (s == "--") break;
    std::string name = s.substr(s[1] == '-' ? 2 : 1), val;
    bool has_val = false;
    size_t eq = name.find('=');
    if (eq != std::string::npos) { val = name.substr(eq + 1); name = name.substr(0, eq); has_val = true; }
    bool done = false;
    for (auto &b : bf)
      if (name == b.name) {
        if (!has_val) *b.dst = true;
        else if (val == "1" || val == "t" || val == "T" || val == "true" || val == "TRUE" || val == "True") *b.dst = true;
        else if (val == "0" || val == "f" || val == "F" || val == "false" || val == "FALSE" || val == "False") *b.dst = false;
        else fatal("invalid boolean value \"" + val + "\" for -" + name);
        done = true;
      }
    if (done) continue;
    std::string *dst = nullptr;
    for (auto &x : sf)
      if (name == x.name) dst = x.dst;
    if (name == "gpus") dst = &gpus;          // extension: number of GPUs to use
    if (name == "chunkBytes") dst = &chunk;   // extension: host chunk size
    if (name == "devices") dst = &devices;    // extension: explicit CUDA device per worker
    if (name == "bgzfLevel") { dst = &level; level_given = true; }  // extension: --bgzfOut's compression level
    if (name == "regions" || name == "regionsFile") {  // extension: region selection
      regions.push_back({name == "regionsFile", ""});
      dst = &regions.back().second;
    }
    if (!dst) fatal("flag provided but not defined: -" + name);
    if (!has_val) {
      if (++i >= argc) fatal("flag needs an argument: -" + name);
      val = argv[i];
    }
    *dst = val;
  }
  if (!allow.empty() && allow != "*") c.allowed = split_trim(allow);  // main.go:108-114
  else c.allowAll = true;
  if (!exclude.empty()) c.excluded = split_trim(exclude);             // main.go:117-123
  if (!gpus.empty()) c.gpus = std::max(1, atoi(gpus.c_str()));
  if (!chunk.empty()) c.chunkBytes = std::max<size_t>(1 << 16, strtoull(chunk.c_str(), nullptr, 10));
  if (!devices.empty()) {
    for (auto &d : split_trim(devices)) c.devices.push_back(atoi(d.c_str()));
    c.gpus = (int)c.devices.size();
  }
  if (level_given) {
    long long v;
    if (!go_int(level, &v)) fatal("invalid value \"" + level + "\" for flag -bgzfLevel: parse error");
    if (v < 1 || v > 9) fatal("--bgzfLevel must be 1..9, not " + std::to_string(v));
    if (!c.bgzfOut) fatal("--bgzfLevel needs --bgzfOut");
    c.bgzfLevel = (int)v;
  }
  for (auto &r : regions) {
    if (r.first) parse_regions_file(r.second, c);
    else parse_regions(r.second, c);
  }
  if (!regions.empty() && c.regionChrom.empty()) fatal("--regionsFile: no intervals");
  c.regionsSet = !regions.empty();
  return c;
}

std::string string_header(const Config &c) {  // main.go:219-239
  bvcf_config k{};
  k.keep_pos = c.keepPos; k.keep_id = c.keepID; k.keep_info = c.keepInfo;
  char buf[512];
  bvcf_header_line(&k, buf, sizeof buf);
  return buf;
}

void write_all(int fd, const uint8_t *p, size_t n) {
  while (n) {
    ssize_t w = write(fd, p, n);
    if (w < 0) {
      if (errno == EINTR) continue;
      fatal(std::string("write: ") + strerror(errno));
    }
    p += w;
    n -= (size_t)w;
  }
}

const char *diag_text(int code) {  // main.go:41-51
  switch (code) {
    case BVCF_DIAG_SAME: return "REF == ALT";
    case BVCF_DIAG_BAD_ALT: return "ALT not ACTG";
    case BVCF_DIAG_DEL1: case BVCF_DIAG_DEL1_LIST: return "1st base REF != ALT";
    case BVCF_DIAG_POS: case BVCF_DIAG_POS_LIST: return "Invalid POS";
    case BVCF_DIAG_INS1: return "1st base ALT != REF";
    case BVCF_DIAG_MIXED: return "Mixed indel/snp sites not supported";
  }
  return "?";
}

// one of the reference's log.Printf lines (main.go:730-986)
void print_diag(const std::string &chrom, const std::string &pos, const bvcf_diag &d) {
  const char *msg = diag_text(d.code);
  switch (d.code) {
    case BVCF_DIAG_SAME: fprintf(stderr, "%s:%s : %s\n", chrom.c_str(), pos.c_str(), msg); break;
    case BVCF_DIAG_MIXED: case BVCF_DIAG_DEL1_LIST:
      fprintf(stderr, "%s:%s ALT#%d %s\n", chrom.c_str(), pos.c_str(), d.alt_no, msg); break;
    case BVCF_DIAG_POS_LIST: fprintf(stderr, "%s:%s %s\n", chrom.c_str(), pos.c_str(), msg); break;
    default: fprintf(stderr, "%s:%s ALT #%d %s\n", chrom.c_str(), pos.c_str(), d.alt_no, msg);
  }
}
// `line` points at the diagnosed line (CHROM \t POS \t ...)
void log_one_diag(const char *line, size_t avail, const bvcf_diag &d) {
  const char *end = line + avail;
  const char *t0 = (const char *)memchr(line, '\t', avail);
  if (!t0) return;
  const char *t1 = (const char *)memchr(t0 + 1, '\t', end - t0 - 1);
  if (!t1) return;
  print_diag(std::string(line, t0), std::string(t0 + 1, t1), d);
}
// the diagnostics of a bgzf chunk, whose text is on the device only: CHROM \t POS of each (bvcf_diag_fields)
void log_diag_fields(const uint8_t *text, const uint64_t *off, const bvcf_diag *d, size_t n) {
  for (size_t k = 0; k < n; k++) {
    const char *f = (const char *)text + off[k];
    const size_t m = (size_t)(off[k + 1] - off[k]);
    const char *t0 = (const char *)memchr(f, '\t', m);
    if (t0) print_diag(std::string(f, t0), std::string(t0 + 1, f + m), d[k]);
  }
}
// the diagnostics of a chunk that is still pinned: every entry carries its line's offset
void log_diags(const uint8_t *chunk, size_t len, const bvcf_diag *d, size_t n) {
  for (size_t k = 0; k < n; k++)
    if (d[k].line_start < len) log_one_diag((const char *)chunk + d[k].line_start, len - d[k].line_start, d[k]);
}

struct Chunk {
  uint64_t seq = 0;
  uint8_t *buf = nullptr;        // pinned buffer holding the chunk (filled by the reader, or by the worker from `src`)
  const uint8_t *src = nullptr;  // memory-mapped input: where the chunk's bytes are
  size_t len = 0;
  // bgzf input: buf holds whole blocks, the chunk's text is inflate(buf)[skip:] + tail (bvcf_submit_bgzf)
  bool gz = false;
  size_t skip = 0;
  std::string tail;
};

// bounded FIFO between the reader and one GPU worker
class ChunkQueue {
 public:
  explicit ChunkQueue(size_t cap) : cap_(cap) {}
  void push(Chunk c) {
    std::unique_lock<std::mutex> l(m_);
    cv_.wait(l, [&] { return q_.size() < cap_; });
    q_.push_back(std::move(c));
    cv_.notify_all();
  }
  void close() {
    std::lock_guard<std::mutex> l(m_);
    closed_ = true;
    cv_.notify_all();
  }
  // 1: got a chunk, 0: nothing right now (only when !block), -1: closed and drained
  int pop(Chunk &c, bool block) {
    std::unique_lock<std::mutex> l(m_);
    if (block) cv_.wait(l, [&] { return !q_.empty() || closed_; });
    if (q_.empty()) return closed_ ? -1 : 0;
    c = std::move(q_.front());
    q_.pop_front();
    cv_.notify_all();
    return 1;
  }

 private:
  std::mutex m_;
  std::condition_variable cv_;
  std::deque<Chunk> q_;
  size_t cap_;
  bool closed_ = false;
};

// a GPU's pinned staging buffers
class BufferPool {
 public:
  void add(uint8_t *b) { std::lock_guard<std::mutex> l(m_); free_.push_back(b); all_.push_back(b); }
  uint8_t *take() {
    std::unique_lock<std::mutex> l(m_);
    cv_.wait(l, [&] { return !free_.empty(); });
    uint8_t *b = free_.back();
    free_.pop_back();
    return b;
  }
  void give(uint8_t *b) { std::lock_guard<std::mutex> l(m_); free_.push_back(b); cv_.notify_all(); }
  ~BufferPool() { for (auto b : all_) bvcf_host_free(b); }

 private:
  std::mutex m_;
  std::condition_variable cv_;
  std::vector<uint8_t *> free_, all_;
};

// whose turn it is to write (chunk order == input order)
struct Turnstile {
  std::mutex m;
  std::condition_variable cv;
  uint64_t next = 0;
  void wait_for(uint64_t seq) { std::unique_lock<std::mutex> l(m); cv.wait(l, [&] { return next == seq; }); }
  void done() { std::lock_guard<std::mutex> l(m); next++; cv.notify_all(); }
};

// ---- bgzf input (.vcf.gz as bgzip / htslib write it): the compressed bytes go to the GPU, which inflates them ----
// Replaces the `pigz -d -c in.vcf.gz |` in front of the reference (README.md:10,46).  Groups of whole blocks are
// uploaded and inflated on the GPU: into a slot's input buffer (bvcf_submit_bgzf), or with --bgzfOut into the resident
// input region (bvcf_resident_inflate_bgzf).
// the input starts with a whole bgzf block header (a first block refused as corrupt is reported by BgzfIn)
bool looks_bgzf(const uint8_t *p, size_t n) {
  size_t bs = 0;
  uint32_t isize;
  const char *why;
  bvcf_bgzf_block(p, n, &bs, &isize, &why);
  return bs > 0;
}

// one bgzf block (SAM spec 4.1) around `text` (< 64 KiB), deflated on the host: the TSV header line
std::vector<uint8_t> bgzf_block_host(const uint8_t *text, size_t n) {
  std::vector<uint8_t> out(18 + compressBound(n) + 8);
  z_stream z{};
  if (deflateInit2(&z, 6, Z_DEFLATED, -15, 8, Z_DEFAULT_STRATEGY) != Z_OK) fatal("deflateInit2 failed");
  z.next_in = const_cast<Bytef *>(text); z.avail_in = (uInt)n;
  z.next_out = out.data() + 18; z.avail_out = (uInt)(out.size() - 18 - 8);
  if (deflate(&z, Z_FINISH) != Z_STREAM_END) fatal("deflate failed");
  const size_t payload = z.total_out;
  deflateEnd(&z);
  const size_t bsize = 18 + payload + 8;
  static const uint8_t hdr[16] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 'B', 'C', 2, 0};
  memcpy(out.data(), hdr, 16);
  out[16] = (uint8_t)((bsize - 1) & 0xFF); out[17] = (uint8_t)((bsize - 1) >> 8);
  const uint32_t crc = (uint32_t)crc32(crc32(0L, Z_NULL, 0), text, (uInt)n), isize = (uint32_t)n;
  for (int k = 0; k < 4; k++) { out[18 + payload + k] = (uint8_t)(crc >> (8 * k)); out[22 + payload + k] = (uint8_t)(isize >> (8 * k)); }
  out.resize(bsize);
  return out;
}
const uint8_t BGZF_EOF[28] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 'B', 'C', 2, 0, 0x1b, 0, 3, 0, 0, 0, 0, 0, 0, 0, 0, 0};

// What main.go:250-294 finds in the first bytes of the text: the EOL width, the #CHROM line, where the data lines start
struct Preamble {
  std::string chrom_line;
  size_t data_off = 0;
  int eol_width = 1;
};

// main.go:250-294 on the first bytes of the text: EOL width, the ##fileformat check, the #CHROM line.  true when found;
// false when more text is needed (fatal at eof)
bool find_preamble(const uint8_t *p, size_t n, bool eof, Preamble &pre) {
  if (n == 0 && eof) fatal("Not a VCF file");
  const uint8_t *nl = (const uint8_t *)memchr(p, '\n', n);
  if (!nl) { if (eof) fatal("Not a VCF file"); return false; }
  size_t first_end = nl - p;
  pre.eol_width = 1;
  if (first_end > 0 && p[first_end - 1] == '\r') { pre.eol_width = 2; first_end--; }
  if (!memmem(p, first_end, "##fileformat=VCFv4", 18)) fatal("Not a VCF file");  // main.go:256-264
  for (size_t q = (nl - p) + 1; q < n;) {
    const uint8_t *e = (const uint8_t *)memchr(p + q, '\n', n - q);
    if (!e) break;
    size_t cl = (e - p) - q;
    cl = cl + 1 >= (size_t)pre.eol_width ? cl + 1 - pre.eol_width : 0;
    if (cl >= 6 && memcmp(p + q, "#CHROM", 6) == 0 && (cl == 6 || p[q + 6] == '\t')) {
      pre.chrom_line.assign((const char *)p + q, cl);
      pre.data_off = (e - p) + 1;
      return true;
    }
    q = (e - p) + 1;
  }
  if (eof) fatal("No header found");  // main.go:293
  return false;
}

// The input bytes: a memory-mapped file, or what has been read from a pipe so far.  Offsets are absolute in the stream.
class Input {
 public:
  Input(int fd, const uint8_t *map, size_t map_len, std::vector<uint8_t> head)
      : fd_(fd), map_(map), map_len_(map_len), buf_(std::move(head)), eof_(map != nullptr) {}
  bool mapped() const { return map_ != nullptr; }
  bool eof() const { return eof_; }
  int fd() const { return fd_; }
  size_t end() const { return map_ ? map_len_ : base_ + buf_.size(); }
  const uint8_t *at(size_t abs) const { return map_ ? map_ + abs : buf_.data() + (abs - base_); }
  void fill(size_t want) {  // bytes up to absolute offset `want` (or the end of the input)
    while (!eof_ && end() < want) {
      const size_t old = buf_.size(), n = std::min<size_t>(8u << 20, std::max<size_t>(want - end(), 1u << 20));
      buf_.resize(old + n);
      const ssize_t r = read(fd_, buf_.data() + old, n);
      if (r < 0) { buf_.resize(old); if (errno == EINTR) continue; fatal(std::string("read: ") + strerror(errno)); }
      buf_.resize(old + (size_t)r);
      if (r == 0) eof_ = true;
    }
  }
  // pipe input: bytes before `abs` are no longer needed
  void release_before(size_t abs) {
    if (map_ || abs - base_ < (64u << 20)) return;
    buf_.erase(buf_.begin(), buf_.begin() + (abs - base_));
    base_ = abs;
  }

 private:
  int fd_;
  const uint8_t *map_;
  size_t map_len_;
  std::vector<uint8_t> buf_;
  size_t base_ = 0;
  bool eof_;
};

// The blocks of a bgzf input, walked as they are needed (pipe input stays bounded in memory).  Blocks without text (the
// EOF block among them) are checked by bvcf_bgzf_block and left out of the list; offsets are absolute in the compressed
// stream.  It is also the block source of bvcf_bgzf_plan.
class BgzfIn {
 public:
  struct Blk { size_t off, size; uint64_t start; uint32_t isize; };
  explicit BgzfIn(Input &in) : in_(in) {}
  // block i exists (reads and walks headers until it does or the input ends; a truncated or corrupt block is fatal)
  bool has(size_t i) {
    while (blk_.size() <= i && !walked_) {
      in_.fill(walk_ + (1u << 16) + 18);  // a whole block, unless the input ends first
      if (walk_ == in_.end()) { walked_ = true; break; }
      size_t bs = 0;
      uint32_t isize = 0;
      const char *why = nullptr;
      if (bvcf_bgzf_block(in_.at(walk_), in_.end() - walk_, &bs, &isize, &why)) fatal(std::string("bgzf input: ") + why);
      if (!bs || walk_ + bs > in_.end()) fatal("bgzf input: truncated block at the end");
      if (isize) blk_.push_back({walk_, bs, text_, isize});
      text_ += isize;
      walk_ += bs;
    }
    return i < blk_.size();
  }
  const Blk &operator[](size_t i) const { return blk_[i]; }
  size_t off(size_t i) { return has(i) ? blk_[i].off : walk_; }  // where block i starts (the end past the last)
  // the first block whose text reaches past text byte `text_off` (the end past the last when none does)
  size_t block_at(uint64_t text_off) {
    size_t b = 0;
    while (has(b) && blk_[b].start + blk_[b].isize <= text_off) b++;
    return b;
  }
  // the first `want` text bytes (fewer at the end of the input), inflated on the host: the preamble
  std::string prefix(size_t want) {
    std::string out;
    for (size_t i = 0; out.size() < want && has(i); i++) {
      const size_t n = out.size();
      const char *why = nullptr;
      out.resize(n + blk_[i].isize);
      if (bvcf_bgzf_inflate(in_.at(blk_[i].off), blk_[i].size, &out[n], blk_[i].isize, &why))
        fatal(std::string("bgzf input: ") + why);
    }
    return out;
  }
  // bvcf_bgzf_block_fn over this input
  static int block(void *self, size_t i, bvcf_bgzf_blk *b) {
    BgzfIn &g = *(BgzfIn *)self;
    if (!g.has(i)) return 0;
    const Blk &k = g.blk_[i];
    *b = {g.in_.at(k.off), k.size, k.start, k.isize};
    return 1;
  }

 private:
  Input &in_;
  size_t walk_ = 0;
  uint64_t text_ = 0;
  bool walked_ = false;
  std::vector<Blk> blk_;
};

// What a run reads: the input from its data lines on -- or, with regions and a tabix / CSI index beside a bgzf input, the
// index's spans only.  A span [vbeg, vend) is a view of the mapped file from the block of vbeg to the end of the block of
// vend, its data lines from vbeg's offset into that first block on; the records after vend in its last block and the
// lines between two regions inside one span are dropped by the GPU's region filter.  Both drivers read these pieces
// through BgzfIn, the streaming one cut into groups by bvcf_bgzf_plan.
struct Piece {
  Input *in;
  BgzfIn *gz;        // null: plain text
  uint64_t data_off;  // text offset of the first data line
};
struct IndexedInput {
  std::vector<std::unique_ptr<Input>> views;
  std::vector<std::unique_ptr<BgzfIn>> gz;
  std::vector<Piece> pieces;
};

// the index file (`<in>.tbi`, else `<in>.csi`) inflated, or empty when there is none
std::string read_index(const std::string &in_path, std::string *which) {
  for (const char *ext : {".tbi", ".csi"}) {
    *which = in_path + ext;
    if (access(which->c_str(), F_OK) != 0) continue;
    gzFile f = gzopen(which->c_str(), "rb");
    if (!f) fatal(*which + ": " + strerror(errno));
    std::string out;
    char buf[1 << 16];
    int n;
    while ((n = gzread(f, buf, sizeof buf)) > 0) out.append(buf, (size_t)n);
    if (n < 0) fatal(*which + ": not a gzip file");
    gzclose(f);
    return out;
  }
  return std::string();
}

// the pieces of a mapped bgzf input that the index of `c.inPath` gives for c's regions; false when there is no index
bool index_pieces(const Config &c, const uint8_t *map, size_t map_len, IndexedInput &out) {
  std::string path;
  const std::string idx = read_index(c.inPath, &path);
  if (idx.empty()) return false;
  std::vector<const char *> names;
  for (auto &s : c.regionChrom) names.push_back(s.c_str());
  std::vector<uint64_t> sp(2 * 1024);
  size_t n = 0;
  int rc = bvcf_index_spans(idx.data(), idx.size(), names.data(), c.regionBeg.data(), c.regionEnd.data(), names.size(),
                            sp.data(), sp.size() / 2, &n);
  if (rc == BVCF_E_TOO_LARGE) {
    sp.resize(2 * n);
    rc = bvcf_index_spans(idx.data(), idx.size(), names.data(), c.regionBeg.data(), c.regionEnd.data(), names.size(),
                          sp.data(), n, &n);
  }
  if (rc) fatal(path + ": " + bvcf_strerror(rc) + " (not a tabix or CSI index)");
  auto size_at = [&](uint64_t off) {  // the size of the bgzf block at compressed offset off; 0 when there is none
    size_t bs = 0;
    uint32_t isize;
    const char *why;
    return off < map_len && !bvcf_bgzf_block(map + off, map_len - off, &bs, &isize, &why) ? (uint64_t)bs : 0;
  };
  auto block_at = [&](uint64_t off) {  // a whole bgzf block starts at compressed offset off: its size
    const uint64_t bs = size_at(off);
    if (!bs || off + bs > map_len)
      fatal(path + ": virtual offset " + std::to_string(off) + " << 16 is not a bgzf block of " + c.inPath);
    return bs;
  };
  for (size_t k = 0; k < n; k++) {
    const uint64_t cb = sp[2 * k] >> 16, ce = sp[2 * k + 1] >> 16, ue = sp[2 * k + 1] & 0xFFFF;
    block_at(cb);
    const uint64_t end = ue ? ce + block_at(ce) : ce;
    if (end < ce || end > map_len || (ce < map_len && !ue && ce != cb && !size_at(ce)))
      fatal(path + ": virtual offset " + std::to_string(ce) + " << 16 is not a bgzf block of " + c.inPath);
    if (end <= cb) continue;
    out.views.emplace_back(new Input(-1, map + cb, (size_t)(end - cb), {}));
    out.gz.emplace_back(new BgzfIn(*out.views.back()));
    out.pieces.push_back({out.views.back().get(), out.gz.back().get(), sp[2 * k] & 0xFFFF});
  }
  return true;
}

// Where the results of a run go (main.go:296-343, 398-445): the rows to the output, the dosage batches to the Arrow
// file.  Built once from the #CHROM line: it writes the sample list and opens the dosage file -- or, when the VCF has no
// samples, writes an empty one and asks for no dosage work.
class Sink {
 public:
  Sink(const Config &c, int out_fd, const std::string &chrom_line) : c_(c), out_fd_(out_fd) {
    std::vector<std::string> names;
    int field = 0;
    size_t s = 0;
    for (size_t i = 0; i <= chrom_line.size(); i++)
      if (i == chrom_line.size() || chrom_line[i] == '\t') {
        if (field >= 9) {
          names.push_back(chrom_line.substr(s, i - s));
          for (auto &ch : names.back()) if (ch == '.') ch = '_';  // parse.NormalizeHeader
        }
        field++; s = i + 1;
      }
    if (!c.sampleListPath.empty() && !c.noOut) {
      FILE *f = fopen(c.sampleListPath.c_str(), "w");
      if (!f) fatal("Couldn't write sample list file");
      for (auto &nm : names) fprintf(f, "%s\n", nm.c_str());
      fclose(f);
    }
#ifndef BVCF_NO_ARROW
    if (c.dosageMatrixOutPath.empty()) return;
    if (names.empty()) {  // main.go:308-318
      fprintf(stderr, "No samples found in VCF file; writing empty dosage matrix file\n");
      FILE *f = fopen(c.dosageMatrixOutPath.c_str(), "w");
      if (!f) fatal(c.dosageMatrixOutPath + ": " + strerror(errno));
      fclose(f);
      return;
    }
    std::vector<const char *> nm;
    for (auto &x : names) nm.push_back(x.c_str());
    char err[512];
    arrow_ = bvcf_arrow_open(c.dosageMatrixOutPath.c_str(), nm.data(), (uint32_t)nm.size(), err, sizeof err);
    if (!arrow_) fatal(std::string("dosage output: ") + err);
#endif
  }
  bool want_dosage() const { return arrow_ != nullptr; }
  void rows(const uint8_t *p, size_t n) {
    if (!c_.noOut) write_all(out_fd_, p, n);
  }
  void dosage(const bvcf_dosage_batch &d) {
#ifndef BVCF_NO_ARROW
    if (arrow_ && d.n_rows && bvcf_arrow_write(arrow_, d.n_rows, d.dosage, d.loci, d.loci_off))
      fatal(std::string("dosage output: ") + bvcf_arrow_error(arrow_));
#endif
  }
  // the exit status: 1 when the Arrow file could not be finished
  int close() {
#ifndef BVCF_NO_ARROW
    if (arrow_ && bvcf_arrow_close(arrow_)) return 1;
#endif
    return 0;
  }

 private:
  const Config &c_;
  int out_fd_;
#ifndef BVCF_NO_ARROW
  bvcf_arrow_writer *arrow_ = nullptr;
#else
  void *arrow_ = nullptr;
#endif
};

// a context on CUDA device `device` for this run, its #CHROM line set
bvcf_ctx *open_ctx(const Config &c, int device, const Preamble &pre, bool want_dosage, int n_slots, size_t max_chunk_bytes) {
  std::vector<const char *> allow_c, excl_c;
  for (auto &s : c.allowed) allow_c.push_back(s.c_str());
  for (auto &s : c.excluded) excl_c.push_back(s.c_str());
  bvcf_config bc{};
  bc.empty_field = c.emptyField.c_str();
  bc.field_delim = c.fieldDelimiter.c_str();
  bc.keep_id = c.keepID; bc.keep_info = c.keepInfo; bc.keep_pos = c.keepPos;
  bc.want_tsv = !c.noOut; bc.want_dosage = want_dosage;
  bc.allow = allow_c.data(); bc.n_allow = c.allowAll ? -1 : (int)allow_c.size();
  bc.exclude = excl_c.data(); bc.n_exclude = (int)excl_c.size();
  bc.eol_width = pre.eol_width; bc.normalize_dots = 1;
  bc.n_slots = n_slots;
  bc.max_chunk_bytes = max_chunk_bytes;
  bvcf_ctx *ctx = nullptr;
  int rc = bvcf_create(&ctx, device, &bc);
  if (rc) fatal(std::string("bvcf_create(gpu ") + std::to_string(device) + "): " + bvcf_strerror(rc) + " -- a CUDA device is required, there is no CPU fallback");
  if ((rc = bvcf_set_header(ctx, pre.chrom_line.data(), pre.chrom_line.size()))) fatal(std::string("bvcf_set_header: ") + bvcf_strerror(rc));
  if (c.regionsSet) {
    std::vector<const char *> names;
    for (auto &s : c.regionChrom) names.push_back(s.c_str());
    if ((rc = bvcf_set_regions(ctx, names.data(), c.regionBeg.data(), c.regionEnd.data(), names.size())))
      fatal(std::string("bvcf_set_regions: ") + bvcf_strerror(rc));
  }
  return ctx;
}

// readVcf for --bgzfOut: the rows are deflated where they are made, so the input goes through one GPU's resident
// regions a group at a time -- plain text uploaded, or whole bgzf blocks inflated there (bvcf_resident_inflate_bgzf).
// The partial line at a group's end is carried into the next group; the one at a piece's end is dropped.
void run_resident(const Config &config, const std::vector<Piece> &pieces, const Preamble &pre, Sink &sink) {
  bvcf_ctx *ctx = open_ctx(config, config.devices.empty() ? 0 : config.devices[0], pre, sink.want_dosage(), 0, 0);
  int rc;
  const size_t batch_text = std::max<size_t>(config.chunkBytes * 8, 64u << 20), max_line = 8u << 20;
  void *d_in, *d_out;
  if ((rc = bvcf_resident_alloc(ctx, batch_text + max_line + (1u << 20), batch_text / 4 + (64u << 20), &d_in, &d_out)))
    fatal(std::string("bvcf_resident_alloc: ") + bvcf_strerror(rc));
  uint8_t *pin = nullptr, *out_host = nullptr;   // pinned: group in, compressed rows out
  size_t pin_cap = 0, out_cap = 0;
  std::vector<uint8_t> carry, tail;
  for (const Piece &piece : pieces) {
    Input &in = *piece.in;
    BgzfIn *gz = piece.gz;
    carry.clear();
    // the first group starts at the data lines (plain) or at the block that holds their first byte (bgzf); `begin` is
    // where they start in it
    size_t pos = piece.data_off, b = 0, begin = 0;
    if (gz && gz->has(b = gz->block_at(piece.data_off))) begin = piece.data_off - (*gz)[b].start;
    for (;;) {
      // ---- a group: whole blocks worth about batch_text bytes of text, or batch_text bytes of plain text ----
      size_t lo = pos, hi;
      if (gz) {
        size_t e = b;
        for (uint64_t text = 0; text < batch_text && gz->has(e); e++) text += (*gz)[e].isize;
        lo = gz->off(b); hi = gz->off(e);  // blocks without text in between go along
        b = e;
      } else {
        in.fill(pos + batch_text);
        hi = pos = std::min(in.end(), pos + batch_text);
      }
      if (hi == lo) break;
      if (hi - lo > pin_cap) {
        if (pin) bvcf_host_free(pin);
        pin_cap = (hi - lo) + (hi - lo) / 4;
        if (bvcf_host_alloc((void **)&pin, pin_cap)) fatal("bvcf_host_alloc failed");
      }
      memcpy(pin, in.at(lo), hi - lo);
      in.release_before(hi);
      if (!carry.empty() && (rc = bvcf_resident_upload(ctx, 0, carry.data(), carry.size()))) fatal(std::string("upload: ") + bvcf_strerror(rc));
      size_t n_text = hi - lo;
      if (gz) {
        if ((rc = bvcf_resident_inflate_bgzf(ctx, pin, hi - lo, carry.size(), &n_text)))
          fatal(std::string("bgzf: ") + bvcf_strerror(rc) + " " + bvcf_last_error(ctx));
      } else if ((rc = bvcf_resident_upload(ctx, carry.size(), pin, hi - lo))) {
        fatal(std::string("upload: ") + bvcf_strerror(rc));
      }
      const size_t total = carry.size() + n_text;
      // ---- the longest newline-terminated prefix; the rest is carried into the next group ----
      const size_t tail_n = std::min(total - begin, max_line);
      tail.resize(tail_n);
      if (tail_n && (rc = bvcf_resident_peek(ctx, total - tail_n, tail.data(), tail_n))) fatal(std::string("peek: ") + bvcf_strerror(rc));
      const uint8_t *last_nl = tail_n ? (const uint8_t *)memrchr(tail.data(), '\n', tail_n) : nullptr;
      if (!last_nl) {
        if (tail_n < total - begin) fatal("a single line exceeds 8 MiB");
        carry.assign(tail.begin(), tail.end());  // no complete line yet: everything is carried
        begin = 0;
        continue;
      }
      const size_t end = total - tail_n + (size_t)(last_nl - tail.data()) + 1;
      bvcf_chunk_stats st{};
      if ((rc = bvcf_resident_run_at(ctx, begin, end, &st, nullptr))) fatal(std::string("bvcf_resident_run: ") + bvcf_strerror(rc) + " " + bvcf_last_error(ctx));
      if (!config.noOut && st.out_bytes) {
        if (st.out_bytes > out_cap) {
          if (out_host) bvcf_host_free(out_host);
          out_cap = st.out_bytes + st.out_bytes / 4;
          if (bvcf_host_alloc((void **)&out_host, out_cap)) fatal("bvcf_host_alloc failed");
        }
        size_t comp = 0;
        rc = bvcf_resident_download_bgzf_level(ctx, 0, st.out_bytes, config.bgzfLevel, out_host, out_cap, &comp);
        if (rc == BVCF_E_TOO_LARGE) {  // comp: the bytes needed
          bvcf_host_free(out_host);
          out_cap = comp + comp / 8;
          if (bvcf_host_alloc((void **)&out_host, out_cap)) fatal("bvcf_host_alloc failed");
          rc = bvcf_resident_download_bgzf_level(ctx, 0, st.out_bytes, config.bgzfLevel, out_host, out_cap, &comp);
        }
        if (rc) fatal(std::string("download: ") + bvcf_strerror(rc) + " " + bvcf_last_error(ctx));
        sink.rows(out_host, comp);
      }
      {  // dosage batch and diagnostics of this group
        bvcf_dosage_batch dos{};
        const bvcf_diag *dg = nullptr;
        size_t nd = 0;
        if ((rc = bvcf_resident_results(ctx, sink.want_dosage() ? &dos : nullptr, &dg, &nd))) fatal(std::string("results: ") + bvcf_strerror(rc));
        sink.dosage(dos);
        char line[4096];
        for (size_t k = 0; k < nd; k++) {
          const size_t n = std::min<size_t>(sizeof line, end - dg[k].line_start);
          if (dg[k].line_start < end && !bvcf_resident_peek(ctx, dg[k].line_start, line, n)) log_one_diag(line, n, dg[k]);
        }
      }
      carry.assign(last_nl + 1, (const uint8_t *)tail.data() + tail_n);
      begin = 0;
    }
  }
  // an unterminated last line (the carry) is dropped (main.go:354-357)
  sink.rows(BGZF_EOF, sizeof BGZF_EOF);
  if (pin) bvcf_host_free(pin);
  if (out_host) bvcf_host_free(out_host);
  bvcf_destroy(ctx);
}

// readVcf on 1..N GPUs: a reader cuts the input into chunks (newline-aligned text, or groups of whole bgzf blocks), chunk
// k goes to GPU k mod N, and each GPU's worker hands its results to the sink when it is the chunk's turn
void run_streaming(const Config &config, const std::vector<Piece> &pieces, const Preamble &pre, Sink &sink) {
  Input &in = *pieces[0].in;
  // ---- one context per GPU ----
  const int n_slots = 3;
  const size_t cap = 2 * config.chunkBytes + (64u << 20);  // a chunk grows until it holds a newline
  const int n_gpu = config.gpus;
  std::vector<bvcf_ctx *> ctxs(n_gpu, nullptr);
  std::vector<BufferPool> pools(n_gpu);
  std::vector<std::unique_ptr<ChunkQueue>> queues;
  for (int g = 0; g < n_gpu; g++) {
    ctxs[g] = open_ctx(config, config.devices.empty() ? g : config.devices[g], pre, sink.want_dosage(), n_slots, cap);
    for (int k = 0; k < n_slots + 2; k++) {
      uint8_t *b = nullptr;
      if (bvcf_host_alloc((void **)&b, cap)) fatal("bvcf_host_alloc failed");
      pools[g].add(b);
    }
    queues.emplace_back(new ChunkQueue(n_slots + 1));
  }

  // ---- GPU workers ----
  Turnstile turn;
  std::mutex fatal_m;
  auto worker = [&](int g) {
    bvcf_ctx *ctx = ctxs[g];
    std::deque<Chunk> inflight;
    bool closed = false;
    for (;;) {
      while (!closed && (int)inflight.size() < n_slots) {
        Chunk c;
        const int got = queues[g]->pop(c, /*block=*/inflight.empty());
        if (got < 0) { closed = true; break; }
        if (got == 0) break;
        if (c.src) {  // memory-mapped input: this thread stages its own chunk (N GPUs, N copies in parallel)
          c.buf = pools[g].take();
          memcpy(c.buf, c.src, c.len);
        }
        const int rc = c.gz ? bvcf_submit_bgzf(ctx, c.seq, c.buf, c.len, c.skip, (const uint8_t *)c.tail.data(), c.tail.size())
                            : bvcf_submit(ctx, c.seq, c.buf, c.len);
        if (rc) { std::lock_guard<std::mutex> l(fatal_m); fatal(std::string("bvcf_submit: ") + bvcf_strerror(rc) + " " + bvcf_last_error(ctx)); }
        inflight.push_back(std::move(c));
      }
      if (inflight.empty()) {
        if (closed) break;
        continue;
      }
      const Chunk c = std::move(inflight.front());
      inflight.pop_front();
      const uint8_t *tsv; size_t n; const bvcf_diag *dg; size_t nd;
      bvcf_dosage_batch dos;
      const int rc = bvcf_collect(ctx, c.seq, &tsv, &n, &dos, &dg, &nd, nullptr);
      int rc2 = 0;
      if (rc) { std::lock_guard<std::mutex> l(fatal_m); fatal(std::string("bvcf_collect: ") + bvcf_strerror(rc) + " " + bvcf_last_error(ctx)); }
      const uint8_t *ftext = nullptr;
      const uint64_t *foff = nullptr;
      if (c.gz && nd && (rc2 = bvcf_diag_fields(ctx, c.seq, &ftext, &foff))) {
        std::lock_guard<std::mutex> l(fatal_m);
        fatal(std::string("bvcf_diag_fields: ") + bvcf_strerror(rc2) + " " + bvcf_last_error(ctx));
      }
      turn.wait_for(c.seq);  // input order
      sink.rows(tsv, n);
      sink.dosage(dos);
      if (c.gz) log_diag_fields(ftext, foff, dg, nd);
      else log_diags(c.buf, c.len, dg, nd);
      turn.done();
      bvcf_release(ctx, c.seq);
      pools[g].give(c.buf);
    }
  };
  std::vector<std::thread> threads;
  for (int g = 0; g < n_gpu; g++) threads.emplace_back(worker, g);

  // ---- reader: newline-aligned chunks, chunk k to GPU k mod N ----
  uint64_t seq = 0;
  if (pieces[0].gz) {  // groups of whole bgzf blocks: a mapped input is staged by the workers, a pipe's by the reader
    for (const Piece &piece : pieces) {
      Input &in = *piece.in;
      BgzfIn *gz = piece.gz;
      auto emit = [&](size_t lo_b, size_t hi_b, size_t skip, const uint8_t *tail, size_t tail_len) {
        const size_t lo = gz->off(lo_b), hi = gz->off(hi_b);
        if (hi - lo > cap) fatal("a bgzf group exceeds the chunk capacity; raise --chunkBytes");
        Chunk c;
        c.seq = seq; c.len = hi - lo; c.gz = true; c.skip = skip; c.tail.assign((const char *)tail, tail_len);
        if (in.mapped()) {
          c.src = in.at(lo);
        } else {
          c.buf = pools[seq % n_gpu].take();
          memcpy(c.buf, in.at(lo), c.len);
          in.release_before(hi);
        }
        queues[seq % n_gpu]->push(std::move(c));
        seq++;
      };
      struct Plan { BgzfIn *gz; decltype(emit) *out; } plan{gz, &emit};
      const char *why = nullptr;
      const int rc = bvcf_bgzf_plan(
          [](void *u, size_t i, bvcf_bgzf_blk *b) { return BgzfIn::block(((Plan *)u)->gz, i, b); },
          [](void *u, size_t lo, size_t hi, size_t skip, const uint8_t *t, size_t n) { (*((Plan *)u)->out)(lo, hi, skip, t, n); return 0; },
          &plan, piece.data_off, config.chunkBytes, cap, &why);
      if (rc) fatal(rc == BVCF_E_ARG && why ? std::string("bgzf input: ") + why : why ? why : bvcf_strerror(rc));
    }
  } else if (in.mapped()) {
    const uint8_t *map = in.at(0);
    size_t p = pre.data_off;
    // an unterminated last line is dropped (main.go:354-357)
    size_t end = in.end();
    {
      const uint8_t *last = end > p ? (const uint8_t *)memrchr(map + p, '\n', end - p) : nullptr;
      end = last ? (size_t)(last - map) + 1 : p;
    }
    while (p < end) {
      size_t q = std::min(p + config.chunkBytes, end);
      if (q < end) {
        const uint8_t *nl = (const uint8_t *)memrchr(map + p, '\n', q - p);
        if (!nl) {  // a line longer than a chunk: extend to its end
          nl = (const uint8_t *)memchr(map + q, '\n', end - q);
          if (!nl) break;
        }
        q = (size_t)(nl - map) + 1;
      }
      if (q - p > cap) fatal("a single line exceeds the chunk capacity; raise --chunkBytes");
      Chunk c;
      c.seq = seq; c.src = map + p; c.len = q - p;
      queues[seq % n_gpu]->push(c);
      seq++;
      p = q;
    }
  } else {  // a pipe is read straight into the pinned buffers, after what the preamble search has read already
    uint8_t *buf = pools[0].take();
    size_t fill = in.end() - pre.data_off;  // bytes already in the current buffer
    if (fill > cap) fatal("header buffer larger than a chunk");
    memcpy(buf, in.at(pre.data_off), fill);
    bool eof = in.eof();
    while (!eof || fill) {
      while (!eof && fill < config.chunkBytes) {
        ssize_t r = read(in.fd(), buf + fill, std::min(cap - fill, config.chunkBytes - fill));
        if (r < 0) { if (errno == EINTR) continue; fatal(std::string("read: ") + strerror(errno)); }
        if (r == 0) { eof = true; break; }
        fill += (size_t)r;
      }
      const uint8_t *last_nl = fill ? (const uint8_t *)memrchr(buf, '\n', fill) : nullptr;
      if (!last_nl) {
        if (eof) break;  // an unterminated last line is dropped (main.go:354-357)
        if (fill >= cap) fatal("a single line exceeds the chunk capacity; raise --chunkBytes");
        ssize_t r = read(in.fd(), buf + fill, cap - fill);
        if (r <= 0) { eof = true; continue; }
        fill += (size_t)r;
        continue;
      }
      const size_t cut = (last_nl - buf) + 1;
      uint8_t *next = pools[(seq + 1) % n_gpu].take();  // the next chunk's buffer comes from its GPU's ring
      memcpy(next, buf + cut, fill - cut);              // carry the partial line
      Chunk c;
      c.seq = seq; c.buf = buf; c.len = cut;
      queues[seq % n_gpu]->push(c);
      seq++;
      fill -= cut;
      buf = next;
    }
    pools[seq % n_gpu].give(buf);
  }
  for (auto &q : queues) q->close();
  for (auto &t : threads) t.join();
  for (auto c : ctxs) bvcf_destroy(c);
}

}  // namespace

int main(int argc, char **argv) {
  Config config = setup(argc, argv);
  int in_fd = 0;
  if (!config.inPath.empty() && (in_fd = open(config.inPath.c_str(), O_RDONLY)) < 0) fatal(config.inPath + ": " + strerror(errno));
  // main.go:150-156 re-points os.Stderr at the file, which Go's `log` never looks at again; what the flag evidently
  // means is honoured here: diagnostics are appended to it
  if (!config.errPath.empty() && !freopen(config.errPath.c_str(), "a", stderr)) fatal(config.errPath + ": " + strerror(errno));
  if (config.noOut && !config.outPath.empty()) fatal("Cannot specify --noOut and --out");                 // main.go:160
  if (config.noOut && config.dosageMatrixOutPath.empty()) fatal("When specifying --noOut, must specify --dosageOutput");  // :164
#ifdef BVCF_NO_ARROW
  if (!config.dosageMatrixOutPath.empty())
    fatal("--dosageOutput: this binary was built without libarrow (pyarrow was not found at build time); "
          "python -m bystro_vcf_b200 writes the Arrow file");
#endif
  int out_fd = 1;
  if (!config.noOut && !config.outPath.empty() &&
      (out_fd = open(config.outPath.c_str(), O_WRONLY | O_CREAT, 0644)) < 0)  // no O_TRUNC, like main.go:172
    fatal(config.outPath + ": " + strerror(errno));
  if (!config.noOut) {
    const std::string h = string_header(config) + "\n";  // main.go:199: before any input is read
    if (config.bgzfOut) {
      const std::vector<uint8_t> b = bgzf_block_host((const uint8_t *)h.data(), h.size());
      write_all(out_fd, b.data(), b.size());
    } else {
      write_all(out_fd, (const uint8_t *)h.data(), h.size());
    }
  }

  // ---- input: a regular file is memory-mapped, anything else (pipes) is read ----
  const uint8_t *map = nullptr;
  size_t map_len = 0;
  struct stat sb;
  if (in_fd != 0 && fstat(in_fd, &sb) == 0 && S_ISREG(sb.st_mode) && sb.st_size > 0) {
    void *m = mmap(nullptr, (size_t)sb.st_size, PROT_READ, MAP_PRIVATE, in_fd, 0);
    if (m != MAP_FAILED) {
      map = (const uint8_t *)m;
      map_len = (size_t)sb.st_size;
      madvise(m, map_len, MADV_SEQUENTIAL);
    }
  }
  std::vector<uint8_t> head;  // pipe input: enough bytes to tell a bgzf input
  if (!map) {
    head.resize(1 << 16);
    size_t got = 0;
    while (got < 18) {
      const ssize_t r = read(in_fd, head.data() + got, head.size() - got);
      if (r < 0) { if (errno == EINTR) continue; fatal(std::string("read: ") + strerror(errno)); }
      if (r == 0) break;
      got += (size_t)r;
    }
    head.resize(got);
  }
  Input in(in_fd, map, map_len, std::move(head));
  std::unique_ptr<BgzfIn> gz;  // .vcf.gz (bgzf) input
  if (looks_bgzf(in.at(0), in.end())) gz.reset(new BgzfIn(in));
  // the rows are deflated where they are, on one GPU's resident regions
  if (config.bgzfOut && config.gpus > 1) fatal("--bgzfOut runs on one GPU");

  // ---- preamble (main.go:250-294): EOL, ##fileformat check, #CHROM line; a bgzf input's is inflated on the host ----
  Preamble pre;
  for (size_t want = 1u << 20;; want *= 4) {
    if (gz) {
      const std::string t = gz->prefix(want);
      if (find_preamble((const uint8_t *)t.data(), t.size(), t.size() < want, pre)) break;
    } else {
      in.fill(want);
      if (find_preamble(in.at(0), in.end(), in.eof(), pre)) break;
    }
  }

  Sink sink(config, out_fd, pre.chrom_line);
  IndexedInput indexed;
  if (!(config.regionsSet && gz && map && index_pieces(config, map, map_len, indexed)))
    indexed.pieces.push_back({&in, gz.get(), pre.data_off});
  if (!indexed.pieces.empty()) {
    if (config.bgzfOut) run_resident(config, indexed.pieces, pre, sink);
    else run_streaming(config, indexed.pieces, pre, sink);
  } else if (config.bgzfOut) {
    sink.rows(BGZF_EOF, sizeof BGZF_EOF);  // no span: no rows
  }
  const int rc_exit = sink.close();
  if (map) munmap((void *)map, map_len);
  if (out_fd != 1) close(out_fd);
  return rc_exit;
}
