// bvcf_index.cpp -- bvcf_index_spans: the bgzf spans a tabix (.tbi) or CSI (.csi) index gives for a set of regions.
// Host only.  Both formats are the binning index of the SAM spec (5.1.1 and 5.2) and of CSIv1.pdf: a bin of level l
// covers 2^(min_shift + 3 (depth - l)) positions, and lists the chunks -- [vbeg, vend) virtual offsets, the compressed
// offset of a bgzf block << 16 | an offset into its text -- that hold records overlapping it.  What a region needs is
// the chunks of every bin that overlaps it, less those that end before the first record that can reach it: the linear
// index (TBI, 16 KiB windows) or the bins' loffset (CSI) says where that record is.
#include <algorithm>
#include <cstring>
#include <map>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/bvcf.h"

namespace {

struct Chunk { uint64_t beg, end; };
struct Bin { uint64_t loff = 0; std::vector<Chunk> chunks; };
struct Ref {
  std::unordered_map<uint32_t, Bin> bins;
  std::vector<uint64_t> lin;  // TBI: the linear index
};
struct Index {
  int min_shift = 14, depth = 5;
  bool csi = false;
  std::map<std::string, size_t> names;
  std::vector<Ref> refs;
};

// a bounds-checked little-endian reader: every read past the end marks the index malformed
struct Rd {
  const uint8_t *p;
  size_t n, i = 0;
  bool bad = false;
  bool has(size_t k) { if (n - i < k) bad = true; return !bad; }
  uint64_t u(int bytes) {
    if (!has((size_t)bytes)) return 0;
    uint64_t v = 0;
    for (int k = 0; k < bytes; k++) v |= (uint64_t)p[i + k] << (8 * k);
    i += (size_t)bytes;
    return v;
  }
  int32_t i32() { return (int32_t)(uint32_t)u(4); }
};

// the contig names of a tabix configuration: l_nm bytes of NUL-terminated names, one per reference
bool read_names(Rd &r, int32_t n_ref, Index &ix) {
  const int32_t l_nm = r.i32();
  if (r.bad || l_nm < 0 || !r.has((size_t)l_nm)) return false;
  const char *s = (const char *)r.p + r.i, *e = s + l_nm;
  for (int32_t k = 0; k < n_ref; k++) {
    const char *z = (const char *)memchr(s, 0, (size_t)(e - s));
    if (!z) return false;
    ix.names.emplace(std::string(s, z), (size_t)k);
    s = z + 1;
  }
  r.i += (size_t)l_nm;
  return true;
}

bool parse(const uint8_t *p, size_t n, Index &ix) {
  Rd r{p, n};
  if (!r.has(4)) return false;
  if (!memcmp(p, "TBI\1", 4)) {
    r.i = 4;
    const int32_t n_ref = r.i32();
    r.u(4 * 6);  // format, col_seq, col_beg, col_end, meta, skip
    if (r.bad || n_ref < 0 || !read_names(r, n_ref, ix)) return false;
    ix.refs.resize((size_t)n_ref);
  } else if (!memcmp(p, "CSI\1", 4)) {
    r.i = 4;
    ix.csi = true;
    ix.min_shift = r.i32();
    ix.depth = r.i32();
    const int32_t l_aux = r.i32();
    if (r.bad || ix.min_shift < 0 || ix.depth < 0 || ix.depth > 10 || ix.min_shift + 3 * ix.depth > 62 || l_aux < 28 || !r.has((size_t)l_aux))
      return false;
    // the aux data of a VCF's CSI index is the tabix configuration: six int32 fields, then the names
    Rd a{p + r.i, (size_t)l_aux};
    r.i += (size_t)l_aux;
    const int32_t n_ref = r.i32();
    a.u(4 * 6);
    if (r.bad || n_ref < 0 || !read_names(a, n_ref, ix)) return false;
    ix.refs.resize((size_t)n_ref);
  } else {
    return false;
  }
  for (auto &ref : ix.refs) {
    const int32_t n_bin = r.i32();
    if (r.bad || n_bin < 0) return false;
    for (int32_t b = 0; b < n_bin; b++) {
      const uint32_t bin = (uint32_t)r.u(4);
      Bin x;
      if (ix.csi) x.loff = r.u(8);
      const int32_t n_chunk = r.i32();
      if (r.bad || n_chunk < 0 || !r.has((size_t)n_chunk * 16)) return false;
      x.chunks.resize((size_t)n_chunk);
      for (auto &c : x.chunks) { c.beg = r.u(8); c.end = r.u(8); }
      ref.bins[bin] = std::move(x);
    }
    if (!ix.csi) {
      const int32_t n_intv = r.i32();
      if (r.bad || n_intv < 0 || !r.has((size_t)n_intv * 8)) return false;
      ref.lin.resize((size_t)n_intv);
      for (auto &v : ref.lin) v = r.u(8);
    }
  }
  return !r.bad;  // an optional count of unplaced records may follow
}

// first bin of level l
uint32_t level_first(int l) { return (uint32_t)(((1ull << (3 * l)) - 1) / 7); }

}  // namespace

extern "C" int bvcf_index_spans(const void *index, size_t len, const char *const *chrom, const int64_t *beg,
                                const int64_t *end, size_t n, uint64_t *spans, size_t cap, size_t *n_spans) {
  if (!index || !n_spans || (n && (!chrom || !beg || !end)) || (cap && !spans)) return BVCF_E_ARG;
  for (size_t i = 0; i < n; i++)
    if (!chrom[i] || !chrom[i][0] || beg[i] < 1 || beg[i] > end[i]) return BVCF_E_ARG;
  Index ix;
  if (!parse((const uint8_t *)index, len, ix)) return BVCF_E_ARG;
  const int s0 = ix.min_shift + 3 * ix.depth;
  const int64_t max_pos = (int64_t)1 << s0;  // positions the binning scheme covers
  // the regions of each contig the file has, merged: a bin shared by many regions is looked at once
  std::map<size_t, std::vector<std::pair<int64_t, int64_t>>> by_ref;
  for (size_t i = 0; i < n; i++) {
    auto it = ix.names.find(chrom[i]);
    if (it != ix.names.end() && beg[i] - 1 < max_pos)  // else a contig the file does not have, or no position it can hold
      by_ref[it->second].push_back({beg[i] - 1, std::min<int64_t>(end[i], max_pos) - 1});  // 0-based, inclusive
  }
  std::vector<std::pair<size_t, std::pair<int64_t, int64_t>>> regs;
  for (auto &kv : by_ref) {
    auto &v = kv.second;
    std::sort(v.begin(), v.end());
    size_t first = regs.size();
    for (auto &x : v) {
      if (regs.size() > first && x.first <= regs.back().second.second + 1) regs.back().second.second = std::max(regs.back().second.second, x.second);
      else regs.push_back({kv.first, x});
    }
  }
  std::vector<Chunk> out;
  for (const auto &rg : regs) {
    const Ref &ref = ix.refs[rg.first];
    const int64_t b0 = rg.second.first, e0 = rg.second.second;
    // the first record that can reach b0 (SAM spec 5.1.3; for CSI the bin loffset, walked as htslib walks it)
    uint64_t min_off = 0;
    if (!ix.csi) {
      if (!ref.lin.empty()) min_off = ref.lin[std::min<size_t>((size_t)(b0 >> ix.min_shift), ref.lin.size() - 1)];
    } else {
      uint32_t bin = level_first(ix.depth) + (uint32_t)(b0 >> ix.min_shift);
      auto f = ref.bins.end();
      for (;;) {
        if ((f = ref.bins.find(bin)) != ref.bins.end() || bin == 0) break;
        const uint32_t first = (((bin - 1) >> 3) << 3) + 1;  // first child of the parent: the first of this level's run
        bin = bin > first ? bin - 1 : (bin - 1) >> 3;
      }
      if (f != ref.bins.end()) min_off = f->second.loff;
    }
    auto take = [&](const Bin &b) {
      for (const Chunk &c : b.chunks)
        if (c.end > min_off && c.end > c.beg) out.push_back(c);
    };
    if ((uint64_t)((e0 >> ix.min_shift) - (b0 >> ix.min_shift)) < ref.bins.size()) {  // the bins overlapping [b0, e0]
      for (int l = 0; l <= ix.depth; l++) {
        const int s = s0 - 3 * l;
        for (int64_t k = b0 >> s; k <= e0 >> s; k++) {
          auto f = ref.bins.find(level_first(l) + (uint32_t)k);
          if (f != ref.bins.end()) take(f->second);
        }
      }
    } else {  // a region wider than the contig's bin list: walk the list (bins past the last level are pseudo-bins)
      for (const auto &kv : ref.bins) {
        int l = 0;
        while (l <= ix.depth && kv.first >= level_first(l + 1)) l++;
        if (l > ix.depth) continue;
        const int s = s0 - 3 * l;
        const int64_t k = (int64_t)(kv.first - level_first(l));
        if (k >= (b0 >> s) && k <= (e0 >> s)) take(kv.second);
      }
    }
  }
  // sorted and merged: overlapping chunks, and chunks that meet in one bgzf block (its text is inflated once)
  std::sort(out.begin(), out.end(), [](const Chunk &a, const Chunk &b) { return a.beg < b.beg; });
  std::vector<Chunk> m;
  for (const Chunk &c : out) {
    if (!m.empty() && (c.beg <= m.back().end || (c.beg >> 16) == (m.back().end >> 16))) m.back().end = std::max(m.back().end, c.end);
    else m.push_back(c);
  }
  *n_spans = m.size();
  if (m.size() > cap) return BVCF_E_TOO_LARGE;
  for (size_t k = 0; k < m.size(); k++) { spans[2 * k] = m[k].beg; spans[2 * k + 1] = m[k].end; }
  return BVCF_OK;
}
