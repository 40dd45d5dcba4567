// bvcf_region.cuh -- the region filter (--regions / --regionsFile): keeps the records whose CHROM is a region's contig
// and whose POS lies in one of its intervals, as an ordered compaction of the input-ordered line table.
//
// It runs only when regions are set, between bvcf_compact_lines_kernel and the genotype summaries; the later stages read
// the kept table and the kept count (RunCounters::chunk_records) and cannot tell the dropped lines were there.  Two
// launches, no host synchronisation:
//   bvcf_region_mark_kernel     a keep byte per record, kept records per block
//   bvcf_region_compact_kernel  each block's base from the block counts, the kept records in input order, the kept count
// Semantics are bcftools view -t (targets): a record is kept when CHROM equals the contig byte for byte and POS is 1 to
// 18 ASCII digits (leading zeros allowed) whose value lies in a [beg, end] interval, 1-based and inclusive.
#pragma once
#include "bvcf_common.cuh"

namespace bvcf {

constexpr int RGN_BLOCKS = 592;  // 4 x 148 SMs
constexpr int RGN_THREADS = 256;

// the regions as the kernels see them: contigs found through an open-addressing hash table, the merged intervals of
// each contig sorted by start and disjoint (bvcf_set_regions builds them)
struct RegionTable {
  const uint8_t *names;       // contig names back to back
  const uint32_t *name_off;   // n_contigs + 1
  const int32_t *slot;        // hash_mask + 1 entries: a contig index, or -1
  uint32_t hash_mask;
  const uint32_t *iv_off;     // n_contigs + 1: the intervals of contig c are [iv_off[c], iv_off[c + 1])
  const long long *beg, *end; // 1-based, inclusive
};

// FNV-1a: the same function on the host (table build) and the device (lookup)
__host__ __device__ __forceinline__ uint32_t region_hash(const uint8_t *s, uint32_t n) {
  uint32_t h = 2166136261u;
  for (uint32_t i = 0; i < n; i++) h = (h ^ s[i]) * 16777619u;
  return h;
}

struct RegionParams {
  const uint8_t *in;
  const LineRec *lines;   // the sub-chunk's input-ordered line table
  LineRec *kept;          // the kept records, in input order
  uint8_t *keep;          // one byte per record
  unsigned int *block_n;  // RGN_BLOCKS + 1: kept records per block, then the sub-chunk's record count
  RegionTable t;
  RunCounters *ctr;
};

__device__ __forceinline__ void rgn_span(uint32_t n, uint32_t &lo, uint32_t &hi) {
  const uint32_t span = (n + RGN_BLOCKS - 1) / RGN_BLOCKS;
  const unsigned long long l = (unsigned long long)blockIdx.x * span;
  lo = l > n ? n : (uint32_t)l;
  hi = l + span > n ? n : (uint32_t)(l + span);
}

// the offset of the first tab at or after `from` (the record has its header's field count: the tab exists)
__device__ __forceinline__ uint32_t rgn_next_tab(const uint8_t *L, uint32_t from, uint32_t n) {
  while (from < n && L[from] != '\t') from++;
  return from;
}

__device__ bool region_keep(const RegionParams &p, const LineRec &rec) {
  const uint8_t *L = p.in + rec.start;
  const uint32_t n = rec.len;
  // CHROM is [0, t0), POS is (t0, t1); a tab past 64 KiB was not recorded by the scan kernel: look for it here
  const uint32_t t0 = rec.tab[0] != 0xFFFFu ? rec.tab[0] : rgn_next_tab(L, 0, n);
  const uint32_t t1 = rec.tab[1] != 0xFFFFu ? rec.tab[1] : rgn_next_tab(L, t0 + 1, n);
  const uint32_t pos_n = t1 - t0 - 1;
  if (t1 <= t0 + 1 || pos_n > 18) return false;
  long long pos = 0;
  for (uint32_t i = 0; i < pos_n; i++) {
    const uint32_t d = (uint32_t)L[t0 + 1 + i] - '0';
    if (d > 9) return false;
    pos = pos * 10 + d;
  }
  const RegionTable &t = p.t;
  int c = -1;
  for (uint32_t h = region_hash(L, t0) & t.hash_mask;; h = (h + 1) & t.hash_mask) {
    const int s = t.slot[h];
    if (s < 0) return false;
    const uint32_t a = t.name_off[s];
    if (t.name_off[s + 1] - a != t0) continue;
    uint32_t i = 0;
    while (i < t0 && t.names[a + i] == L[i]) i++;
    if (i == t0) { c = s; break; }
  }
  // the last interval that starts at or before pos
  uint32_t lo = t.iv_off[c], hi = t.iv_off[c + 1];
  while (lo < hi) {
    const uint32_t mid = (lo + hi) >> 1;
    if (t.beg[mid] <= pos) lo = mid + 1;
    else hi = mid;
  }
  return lo > t.iv_off[c] && pos <= t.end[lo - 1];
}

__global__ void __launch_bounds__(RGN_THREADS) bvcf_region_mark_kernel(const RegionParams p) {
  __shared__ unsigned int sh[RGN_THREADS / 32];
  const uint32_t n = p.ctr->chunk_records;
  uint32_t lo, hi;
  rgn_span(n, lo, hi);
  unsigned int kept = 0;
  for (uint32_t i = lo + threadIdx.x; i < hi; i += RGN_THREADS) {
    const bool k = region_keep(p, p.lines[i]);
    p.keep[i] = k;
    kept += k;
  }
  kept = warp_sum(kept);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = kept;
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned int s = 0;
    for (int w = 0; w < RGN_THREADS / 32; w++) s += sh[w];
    p.block_n[blockIdx.x] = s;
    // the next kernel rewrites chunk_records: it takes the record count from here
    if (blockIdx.x == 0) p.block_n[RGN_BLOCKS] = n;
  }
}

__global__ void __launch_bounds__(RGN_THREADS) bvcf_region_compact_kernel(const RegionParams p) {
  __shared__ unsigned int sh[RGN_THREADS / 32];
  __shared__ unsigned int s_base;
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  const uint32_t n = p.block_n[RGN_BLOCKS];
  // kept records of the blocks before this one (the last block counts its own too: that is the kept count)
  const uint32_t upto = blockIdx.x == RGN_BLOCKS - 1 ? RGN_BLOCKS : blockIdx.x;
  unsigned int b = 0;
  for (uint32_t j = threadIdx.x; j < upto; j += RGN_THREADS) b += p.block_n[j];
  b = warp_sum(b);
  if (l == 0) sh[w] = b;
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned int s = 0;
    for (int k = 0; k < RGN_THREADS / 32; k++) s += sh[k];
    s_base = blockIdx.x == RGN_BLOCKS - 1 ? s - p.block_n[blockIdx.x] : s;
    if (blockIdx.x == RGN_BLOCKS - 1) p.ctr->chunk_records = s;
  }
  __syncthreads();
  unsigned int base = s_base;
  uint32_t lo, hi;
  rgn_span(n, lo, hi);
  for (uint32_t i0 = lo; i0 < hi; i0 += RGN_THREADS) {
    const uint32_t i = i0 + threadIdx.x;
    const uint32_t k = i < hi ? p.keep[i] : 0u;
    const uint32_t incl = warp_incl_scan(k, l);
    __syncthreads();  // sh is read below by the previous round
    if (l == 31) sh[w] = incl;
    __syncthreads();
    unsigned int before = 0, total = 0;
#pragma unroll
    for (int q = 0; q < RGN_THREADS / 32; q++) {
      if (q < w) before += sh[q];
      total += sh[q];
    }
    if (k) p.kept[base + before + incl - 1] = p.lines[i];
    base += total;
  }
}

}  // namespace bvcf
