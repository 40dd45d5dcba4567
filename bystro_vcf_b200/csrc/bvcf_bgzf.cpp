// bvcf_bgzf.cpp -- bgzf input on the host, once for both hosts (bvcf_host.cpp and bystro_vcf_b200/bgzf.py): the block
// header rule, the host inflate of a block, and the plan that cuts an input into groups of whole blocks for
// bvcf_submit_bgzf.  Host only; the DEFLATE payloads of the groups are inflated on the GPU (bvcf_inflate.cuh).
#include <deque>
#include <new>
#include <string>

#include <zlib.h>

#include "../../include/bvcf.h"
#include "bvcf_bgzf.h"

static uint32_t le32(const uint8_t *p) {
  return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
}

// A gzip member with FLG.FEXTRA whose extra field holds a BC subfield with SLEN 2 -- anywhere in the field (SAM spec
// 4.1).  The subfields are walked in order, one that runs past the end of the field ends the walk, and the first BC
// subfield gives BSIZE - 1.
long long bgzf_header(const uint8_t *p, size_t n, const char **why) {
  const char *w = nullptr;
  if (n < 18) return 0;
  if (p[0] != 0x1f || p[1] != 0x8b || p[2] != 8 || !(p[3] & 4)) {
    w = "not a bgzf block";
  } else {
    const size_t xlen = (size_t)p[10] | ((size_t)p[11] << 8);
    if (n < 12 + xlen) return 0;
    w = "gzip member without the bgzf BC subfield (plain gzip: decompress it first, gzip -dc | ...)";
    for (size_t q = 12; q + 4 <= 12 + xlen;) {
      const size_t slen = (size_t)p[q + 2] | ((size_t)p[q + 3] << 8);
      if (q + 4 + slen > 12 + xlen) break;
      if (p[q] == 'B' && p[q + 1] == 'C' && slen == 2) {
        const size_t bsize = ((size_t)p[q + 4] | ((size_t)p[q + 5] << 8)) + 1;
        if (bsize >= 12 + xlen + 8) return (long long)bsize;
        w = "bgzf block smaller than its header and trailer";
        break;
      }
      q += 4 + slen;
    }
  }
  if (why) *why = w;
  return -1;
}

int bvcf_bgzf_inflate(const void *block, size_t n, void *text, size_t cap, const char **why) {
  const uint8_t *p = (const uint8_t *)block;
  const char *w = nullptr;
  const long long bs = p ? bgzf_header(p, n, &w) : -1;
  if (bs <= 0 || (size_t)bs > n) {
    if (why) *why = w ? w : "truncated bgzf block";
    return BVCF_E_ARG;
  }
  const size_t xlen = (size_t)p[10] | ((size_t)p[11] << 8);
  const uint32_t crc = le32(p + bs - 8), isize = le32(p + bs - 4);
  if (isize > cap) return BVCF_E_TOO_LARGE;
  uint8_t none;
  Bytef *out = isize ? (Bytef *)text : &none;  // zlib refuses a null output buffer, even for no bytes
  z_stream z{};
  if (inflateInit2(&z, -15) != Z_OK) return BVCF_E_NOMEM;
  z.next_in = const_cast<Bytef *>(p + 12 + xlen); z.avail_in = (uInt)(bs - 12 - xlen - 8);
  z.next_out = out; z.avail_out = isize;
  const int zr = inflate(&z, Z_FINISH);
  const size_t got = z.total_out;
  inflateEnd(&z);
  if (zr != Z_STREAM_END || got != isize || crc32(crc32(0L, Z_NULL, 0), out, (uInt)got) != crc) {
    if (why) *why = "corrupt bgzf block (inflate, CRC-32 or ISIZE check failed)";
    return BVCF_E_ARG;
  }
  return BVCF_OK;
}

int bvcf_bgzf_block(const void *p, size_t n, size_t *size, uint32_t *isize, const char **why) {
  if (!p || !size || !isize) return BVCF_E_ARG;
  const long long bs = bgzf_header((const uint8_t *)p, n, why);
  if (bs < 0) return BVCF_E_ARG;
  *size = (size_t)bs;
  if (bs == 0 || (size_t)bs > n) return BVCF_OK;
  *isize = le32((const uint8_t *)p + bs - 4);
  // a block that claims no text (normally the 28-byte EOF block) is inflated: text behind it would be dropped unseen
  return *isize ? BVCF_OK : bvcf_bgzf_inflate(p, n, nullptr, 0, why);
}

int bvcf_bgzf_blocks(const void *p, size_t n, uint32_t *size, uint32_t *isize, size_t cap, size_t *n_blocks,
                     const char **why) {
  if (!p || !size || !isize || !n_blocks) return BVCF_E_ARG;
  size_t k = 0, at = 0, bs = 0;
  int rc = BVCF_OK;
  for (; k < cap; k++, at += bs) {
    if ((rc = bvcf_bgzf_block((const uint8_t *)p + at, n - at, &bs, &isize[k], why))) break;
    if (!bs || bs > n - at) break;
    size[k] = (uint32_t)bs;
  }
  *n_blocks = k;
  return rc;
}

namespace {

struct Stop { int rc; const char *why; };  // ends the plan: a refusal, or what a callback returned

struct Planner {
  bvcf_bgzf_block_fn block_fn;
  bvcf_bgzf_emit_fn emit_fn;
  void *user;
  size_t cap;
  struct G { size_t lo, hi, skip; std::string tail; bool set = false; } prev;  // the group held back

  // the blocks asked for so far from block `first` on (those before the held-back group are not read again); their
  // bytes are asked for again before they are read
  std::deque<bvcf_bgzf_blk> blk;
  size_t first = 0;
  bool ended = false;

  bool has(size_t i) {
    while (first + blk.size() <= i && !ended) {
      bvcf_bgzf_blk b{};
      const int r = block_fn(user, first + blk.size(), &b);
      if (r < 0) throw Stop{r, nullptr};
      if (r == 0) ended = true;
      else blk.push_back(b);
    }
    return i < first + blk.size();
  }
  const bvcf_bgzf_blk &at(size_t i) { return blk[i - first]; }  // block i, after has(i)
  std::string text(size_t i) {  // block i inflated on the host
    bvcf_bgzf_blk b{};
    const int r = block_fn(user, i, &b);
    if (r <= 0) throw Stop{r < 0 ? r : BVCF_E_STATE, nullptr};
    std::string t(b.isize, '\0');
    const char *why = nullptr;
    if (const int rc = bvcf_bgzf_inflate(b.bytes, b.size, &t[0], t.size(), &why)) throw Stop{rc, why};
    return t;
  }
  uint64_t text_of(size_t lo, size_t hi) { return hi == lo ? 0 : at(hi - 1).start + at(hi - 1).isize - at(lo).start; }
  size_t take(size_t i, size_t chunk_bytes) {  // the end block of the group candidate that starts at block i
    size_t e = i;
    while (has(e) && at(e).start - at(i).start < chunk_bytes) e++;
    return e;
  }
  void line_too_long() { throw Stop{BVCF_E_TOO_LARGE, "a single line exceeds the chunk capacity; raise --chunkBytes"}; }
  void out(const G &g) {
    if (const int r = emit_fn(user, g.lo, g.hi, g.skip, (const uint8_t *)g.tail.data(), g.tail.size())) throw Stop{r, nullptr};
  }
  void emit(size_t lo, size_t hi, size_t skip, std::string tail) {
    const uint64_t t = text_of(lo, hi);
    if (t + tail.size() > cap) line_too_long();
    if (t - skip + tail.size() == 0) return;
    if (prev.set) out(prev);
    prev = G{lo, hi, skip, std::move(tail), true};
    for (; first < lo; first++) blk.pop_front();
  }

  void run(uint64_t data_off, size_t chunk_bytes) {
    size_t b = 0;
    while (has(b) && at(b).start + at(b).isize <= data_off) b++;
    if (!has(b)) return;
    size_t skip = (size_t)(data_off - at(b).start);
    for (;;) {
      size_t e = take(b, chunk_bytes);
      bool found = false;
      std::string tail;
      while (has(e) && !found) {
        const size_t e2 = take(e, chunk_bytes);
        tail.clear();
        for (size_t j = e; j < e2 && !found; j++) {  // the continuation: inflated until its newline
          const std::string t = text(j);
          const size_t k = t.find('\n');
          if (k != std::string::npos) { tail.append(t, 0, k + 1); found = true; }
          else tail += t;
        }
        if (!found) e = e2;  // no newline in the next group: it joins this one
      }
      if (found) {
        const size_t n = tail.size();
        emit(b, e, skip, std::move(tail));
        b = e; skip = n;
        continue;
      }
      // the last group [b, e): it ends at the input's last newline
      size_t f = e;
      std::string last;
      bool nl = false;
      while (f > b && !nl) {
        const std::string t = text(--f);
        const size_t k = t.rfind('\n');
        if (k != std::string::npos) { last.assign(t, 0, k + 1); nl = true; }
      }
      if (nl) {
        const uint64_t data_start = at(b).start + skip, f_start = at(f).start;
        if (data_start < f_start) {
          emit(b, f, skip, std::move(last));
        } else if (data_start - f_start < last.size()) {  // the rest is inside the block of the last newline
          std::string rest = last.substr((size_t)(data_start - f_start));
          if (prev.set) {
            prev.tail += rest;  // the previous group's tail takes it
            if (text_of(prev.lo, prev.hi) + prev.tail.size() > cap) line_too_long();
          } else {
            emit(f, f, 0, std::move(rest));
          }
        }
      }
      if (prev.set) out(prev);
      return;
    }
  }
};

}  // namespace

int bvcf_bgzf_plan(bvcf_bgzf_block_fn block, bvcf_bgzf_emit_fn emit, void *user, uint64_t data_off, size_t chunk_bytes,
                   size_t cap, const char **why) {
  if (!block || !emit) return BVCF_E_ARG;
  try {
    Planner{block, emit, user, cap}.run(data_off, chunk_bytes);
  } catch (const Stop &s) {
    if (why && s.why) *why = s.why;
    return s.rc;
  } catch (const std::bad_alloc &) {
    return BVCF_E_NOMEM;
  }
  return BVCF_OK;
}
