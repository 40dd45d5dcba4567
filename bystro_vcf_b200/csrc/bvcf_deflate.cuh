// bvcf_deflate.cuh -- SURVEY 8f-4: output-side compression on the GPU.  The reference's pipeline ends in
// `| pigz -c > out.gz` (README.md:10,71): here the TSV rows can leave the device already as bgzf (block gzip: what
// bgzip / htslib write and any gunzip reads), so that the compressed bytes cross PCIe and no host core deflates.
//
// One warp per 48 KiB slice of the output buffer (slices ignore row boundaries: gzip members concatenate).
//   * LZ77: 32 positions per step, one per lane.  A lane hashes its four bytes into a 4,096-entry table of last
//     positions (shared memory), verifies the candidate byte by byte (up to 258), and the warp takes matches greedily
//     in position order (ballot / ffs); the positions in between are literals.
//   * Encoding: DEFLATE fixed Huffman codes (RFC 1951 3.2.6) -- no tree to build or ship; every lane knows its token's
//     bits, a warp prefix sum places them, and they are OR-ed into the (zeroed) output words with reductions
//     (RED.OR: fire and forget).
//   * CRC-32 of the slice (gzip's trailer): crc_warp (bvcf_crc.cuh), each lane a 1.5 KiB run.
// bvcf_deflate_pack_kernel then moves the blocks, now of known size, back to back.
// bvcf_deflate_kernel is level 1, a throughput-first compressor (single candidate per hash, no lazy matching, fixed
// codes): sample-name lists deflate about 2.3x with it where `gzip -6` reaches 3-4x.
//
// Levels 2..9 (bvcf_deflate_dyn_kernel, same slices, same members, same pack kernel):
//   * LZ77 with a bounded search: each hash bucket keeps its last `cands` positions (DEF_LEVELS), a lane tries them
//     and the earlier lanes of its step with the same hash, and takes the longest verified match in 32 KiB; from level
//     4 on, one-step lazy matching.  The positions of a step enter the table in lane order, so the output is the same
//     on every run.
//   * The pass runs twice: once to count the literal/length and distance symbols, once to emit them, so that no token
//     stream is kept.  In between, one warp builds length-limited canonical Huffman codes (15 bits; 7 for the
//     code-length code) and the dynamic block header, and takes the cheapest of dynamic, fixed and stored by exact
//     bit count: a member never exceeds the stored size, 18 + 5 + 49,152 + 8 bytes.
//   * Bits are placed as at level 1 (warp prefix sum, OR into zeroed words); CRC-32 through crc_warp.
//   ptxas (sm_100a): 64 registers, 3,248 B of static shared memory plus the hash table in dynamic shared memory (it
//   holds the code builder's scratch between the passes), a 160 B stack frame for lane 0's small arrays, no spills.
//   Shared memory sets the CTAs (warps) per SM: 11 with the 16 KiB table of levels 3..6, 7 with 32 KiB (levels 8, 9).
#pragma once
#include "bvcf_common.cuh"
#include "bvcf_crc.cuh"

namespace bvcf {

constexpr uint32_t DEF_SLICE = 49152;                       // text bytes per bgzf block
constexpr uint32_t DEF_SLOT = 57376;                        // >= 18 + 49152 * 9 / 8 + 1 + 8 (header, 9 bits per byte, end code, trailer), a multiple of 16
constexpr uint32_t DEF_HASH_BITS = 12;
constexpr uint32_t DEF_MIN_MATCH = 4, DEF_MAX_MATCH = 258;

struct DeflateParams {
  const uint8_t *text;          // the rows
  unsigned long long text_len;
  uint8_t *slots;               // n_blocks x DEF_SLOT, zeroed
  uint32_t *sizes;              // bytes of each finished block
  uint32_t n_blocks;
};

// the bits of one DEFLATE token, LSB first, and their count (at most 31)
__device__ __forceinline__ uint32_t def_rev(uint32_t code, int bits) { return __brev(code) >> (32 - bits); }
__device__ __forceinline__ uint32_t def_literal(uint32_t c, int &n) {
  if (c < 144) { n = 8; return def_rev(0x30u + c, 8); }
  n = 9;
  return def_rev(0x190u + (c - 144u), 9);
}
__device__ __forceinline__ uint32_t def_match(uint32_t len, uint32_t dist, int &n) {
  uint32_t bits;
  int nb;
  {  // length code 257..285 + extra bits
    const uint32_t l = len - 3u;
    uint32_t code, ev = 0;
    int e = 0;
    if (len == 258u) code = 285u;
    else if (l < 8u) code = 257u + l;
    else {
      const int b = 31 - __clz(l);
      e = b - 2;
      code = 265u + 4u * (uint32_t)(e - 1) + ((l >> e) & 3u);
      ev = l & ((1u << e) - 1u);
    }
    if (code < 280u) { bits = def_rev(code - 256u, 7); nb = 7; }
    else { bits = def_rev(0xC0u + (code - 280u), 8); nb = 8; }
    bits |= ev << nb; nb += e;
  }
  {  // distance code 0..29 (5 bits) + extra bits
    const uint32_t t = dist - 1u;
    uint32_t code, ev = 0;
    int e = 0;
    if (t < 4u) code = t;
    else {
      const int b = 31 - __clz(t);
      e = b - 1;
      code = 2u * (uint32_t)b + ((t >> e) & 1u);
      ev = t & ((1u << e) - 1u);
    }
    bits |= def_rev(code, 5) << nb; nb += 5;
    bits |= ev << nb; nb += e;
  }
  n = nb;
  return bits;
}

__global__ void __launch_bounds__(32) bvcf_deflate_kernel(const DeflateParams p) {
  __shared__ unsigned short s_hash[1u << DEF_HASH_BITS];
  __shared__ uint32_t s_crc[256];
  const int lane = threadIdx.x;
  const uint32_t bi = blockIdx.x;
  if (bi >= p.n_blocks) return;
  const unsigned long long t0 = (unsigned long long)bi * DEF_SLICE;
  const uint32_t len = (uint32_t)(p.text_len - t0 < DEF_SLICE ? p.text_len - t0 : DEF_SLICE);
  const uint8_t *in = p.text + t0;
  uint8_t *slot = p.slots + (size_t)bi * DEF_SLOT;
  // the DEFLATE bits start at byte 18: stream bit b lives in bit (b + 16) % 32 of word (b + 16) / 32 of this view
  uint32_t *sw = reinterpret_cast<uint32_t *>(slot + 16);
  for (int i = lane; i < (1 << DEF_HASH_BITS); i += 32) s_hash[i] = 0;
  crc_table_init(s_crc, lane);
  __syncwarp();

  const uint32_t crc = crc_warp([&](uint32_t i) { return (uint32_t)in[i]; }, len, lane, s_crc);

  // ---- LZ77 + fixed Huffman ----
  uint32_t bitpos = 3;   // BFINAL = 1, BTYPE = 01 (fixed codes): bits 1, 1, 0 -> value 3, written with the header below
  uint32_t cur = 0;      // first position not covered by a token yet
  for (uint32_t base = 0; base < len; base += 32) {
    const uint32_t pos = base + lane;
    uint32_t mlen = 0, mdist = 0, c0 = 0;
    if (pos < len) {
      c0 = in[pos];
      if (pos + 4 <= len) {
        const uint32_t w = (uint32_t)in[pos] | ((uint32_t)in[pos + 1] << 8) | ((uint32_t)in[pos + 2] << 16) | ((uint32_t)in[pos + 3] << 24);
        const uint32_t h = (w * 2654435761u) >> (32 - DEF_HASH_BITS);
        // position + 1 of an earlier occurrence of (probably) these four bytes; a lane may also see what another lane
        // of this step has just written: later positions are rejected below
        const uint32_t cand = s_hash[h];
        s_hash[h] = (unsigned short)(pos + 1);  // slices are 48 KiB: positions fit 16 bits
        if (cand && cand - 1 < pos && pos - (cand - 1) <= 32768u && pos >= cur) {
          const uint8_t *a = in + (cand - 1), *b = in + pos;
          const uint32_t lim = len - pos < DEF_MAX_MATCH ? len - pos : DEF_MAX_MATCH;
          uint32_t n = 0;
          while (n < lim && a[n] == b[n]) n++;
          if (n >= DEF_MIN_MATCH) { mlen = n; mdist = pos - (cand - 1); }
        }
      }
    }
    __syncwarp();
    // greedy, in position order: the first lane at or after `cur` with a match takes it, the lanes before it are literals
    uint32_t c = cur > base ? cur - base : 0u;   // step-local cursor (may start beyond 31: the whole step is covered)
    uint32_t role = 0;                            // 0 covered, 1 literal, 2 match
    const uint32_t n_here = len - base < 32u ? len - base : 32u;
    while (c < n_here) {
      const uint32_t mm = __ballot_sync(FULL, mlen != 0 && (uint32_t)lane >= c && (uint32_t)lane < n_here);
      const uint32_t f = mm ? (uint32_t)(__ffs(mm) - 1) : n_here;
      if ((uint32_t)lane >= c && (uint32_t)lane < f) role = 1;
      if (f >= n_here) { c = n_here; break; }
      if ((uint32_t)lane == f) role = 2;
      c = f + __shfl_sync(FULL, mlen, (int)f);
    }
    cur = base + c;
    int nb = 0;
    uint32_t bits = 0;
    if (role == 1) bits = def_literal(c0, nb);
    else if (role == 2) bits = def_match(mlen, mdist, nb);
    const uint32_t incl = warp_incl_scan((uint32_t)nb, lane);
    if (nb) {
      const uint32_t at = bitpos + incl - (uint32_t)nb + 16u;      // bit offset in the word view
      const unsigned long long v = (unsigned long long)bits << (at & 31u);
      atomicOr(sw + (at >> 5), (uint32_t)v);
      if ((uint32_t)(v >> 32)) atomicOr(sw + (at >> 5) + 1, (uint32_t)(v >> 32));
    }
    bitpos += __shfl_sync(FULL, incl, 31);
  }
  // end-of-block code: seven zero bits (nothing to OR), then pad to a byte
  bitpos += 7;
  const uint32_t dbytes = (bitpos + 7u) >> 3;
  const uint32_t total = 18u + dbytes + 8u;
  __syncwarp();
  if (lane == 0) {
    // gzip member header with the bgzf extra field (SAM spec 4.1); bytes 16, 17 hold BSIZE - 1 and share a word with
    // the first stream bits: OR them in
    const uint8_t hdr[16] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 'B', 'C', 2, 0};
    for (int i = 0; i < 16; i++) slot[i] = hdr[i];
    atomicOr(sw, ((total - 1u) & 0xFFFFu) | (3u << 16));   // BSIZE - 1, then BFINAL = 1 / BTYPE = 01
    p.sizes[bi] = total;
  }
  __syncwarp();
  __threadfence_block();
  if (lane == 0) {
    uint8_t *t = slot + 18 + dbytes;  // the reductions above are to global memory of this very thread block's slot; the
                                      // trailer bytes are disjoint from every word they touch except possibly the last
    const uint32_t tr[2] = {crc, len};
    // byte-granular ORs through the word view keep the last stream word intact
    for (int k = 0; k < 8; k++) {
      const uint32_t byte = (tr[k >> 2] >> (8 * (k & 3))) & 0xFFu;
      uint8_t *q = t + k;
      uint32_t *qw = reinterpret_cast<uint32_t *>((uintptr_t)q & ~(uintptr_t)3);
      atomicOr(qw, byte << (8 * ((uintptr_t)q & 3u)));
    }
  }
}

// ---- levels 2..9: bvcf_deflate_dyn_kernel ------------------------------------------------------------------------
// The search of each level: `cands` positions kept per hash bucket (the most recent first) and tried at every position,
// the longest verified match within 32 KiB taken; from level 4 on (where zlib starts matching lazily) a match is given
// up for a literal when the next position has a longer one.  Level 1 is bvcf_deflate_kernel (its row is not read).
// A table has (1 << hash_bits) * cands entries of 2 bytes, in dynamic shared memory (def_dyn_smem): the kernel is
// latency-bound, so the table's size sets how many slices an SM works on at once -- 16 KiB up to level 6.
struct DeflateLevel {
  uint8_t cands, hash_bits, lazy;
};
constexpr DeflateLevel DEF_LEVELS[10] = {
    {0, 0, 0},  {1, 12, 0}, {1, 12, 0}, {2, 12, 0}, {2, 12, 1},
    {3, 11, 1}, {4, 11, 1}, {6, 11, 1}, {8, 11, 1}, {8, 11, 1}};
constexpr uint32_t DEF_WINDOW = 32768;
constexpr uint32_t DEF_NLIT = 286, DEF_NDIST = 30, DEF_NPRE = 19;
// the words of a slot the stream may touch (the DEFLATE bits start at byte 18; the word view starts at byte 16)
constexpr uint32_t DEF_SLOT_WORDS = (DEF_SLOT - 16) / 4;

// length 3..258 -> symbol index 0..28 (symbol 257 + index) and its extra bits; distance 1..32768 -> code 0..29 and its
// extra bits (RFC 1951 3.2.5; the same arithmetic as def_match)
__device__ __forceinline__ uint32_t def_len_sym(uint32_t len, uint32_t &ev, uint32_t &e) {
  const uint32_t l = len - 3u;
  ev = 0; e = 0;
  if (len == 258u) return 28u;
  if (l < 8u) return l;
  const uint32_t b = 31u - __clz(l);
  e = b - 2u;
  ev = l & ((1u << e) - 1u);
  return 8u + 4u * (e - 1u) + ((l >> e) & 3u);
}
__device__ __forceinline__ uint32_t def_dist_sym(uint32_t dist, uint32_t &ev, uint32_t &e) {
  const uint32_t t = dist - 1u;
  ev = 0; e = 0;
  if (t < 4u) return t;
  const uint32_t b = 31u - __clz(t);
  e = b - 1u;
  ev = t & ((1u << e) - 1u);
  return 2u * b + ((t >> e) & 1u);
}
__host__ __device__ __forceinline__ uint32_t def_len_extra(uint32_t i) { return (i < 8u || i == 28u) ? 0u : (i - 4u) / 4u; }
__host__ __device__ __forceinline__ uint32_t def_dist_extra(uint32_t d) { return d < 4u ? 0u : d / 2u - 1u; }
__host__ __device__ __forceinline__ uint32_t def_fixed_llen(uint32_t s) { return s < 144u ? 8u : s < 256u ? 9u : s < 280u ? 7u : 8u; }

// four text bytes from any address; the word after an aligned one is not read (it may lie past the buffer)
__device__ __forceinline__ uint32_t def_ld32(const uint8_t *p) {
  const uintptr_t a = (uintptr_t)p;
  const uint32_t *w = reinterpret_cast<const uint32_t *>(a & ~(uintptr_t)3);
  const uint32_t sh = (uint32_t)(a & 3u) * 8u;
  const uint32_t lo = __ldg(w);
  return sh ? __funnelshift_r(lo, __ldg(w + 1), sh) : lo;
}

// the longest match for `pos` among its candidates: first the earlier lanes of this step with the same hash (`lower`,
// nearest first), then the bucket's row; the nearest of equally long matches wins.  0 when shorter than 4.
__device__ __forceinline__ void def_longest(const uint8_t *in, uint32_t len, uint32_t pos, uint32_t base, uint32_t lower,
                                            const unsigned short *row, int k, uint32_t &mlen, uint32_t &mdist) {
  const uint32_t lim = len - pos < DEF_MAX_MATCH ? len - pos : DEF_MAX_MATCH;
  uint32_t best = 0, bdist = 0;
  int j = 0;
#pragma unroll 1
  for (int t = 0; t < k; t++) {
    uint32_t cand;
    if (lower) {
      const uint32_t l = 31u - __clz(lower);
      lower ^= 1u << l;
      cand = base + l;
    } else {
      const uint32_t e = row[j++];
      if (!e) break;
      cand = e - 1u;
    }
    const uint32_t dist = pos - cand;
    if (dist > DEF_WINDOW) break;                        // the rest are older still
    if (best && in[cand + best] != in[pos + best]) continue;  // cannot be longer
    const uint8_t *a = in + cand, *b = in + pos;
    uint32_t n = 0;
    while (n + 4u <= lim) {
      const uint32_t x = def_ld32(a + n) ^ def_ld32(b + n);
      if (x) { n += (uint32_t)(__ffs(x) - 1) >> 3; goto done; }
      n += 4u;
    }
    while (n < lim && a[n] == b[n]) n++;
  done:
    if (n > best) {
      best = n; bdist = dist;
      if (n == lim) break;
    }
  }
  if (best >= DEF_MIN_MATCH) { mlen = best; mdist = bdist; }
  else { mlen = 0; mdist = 0; }
}

__device__ __forceinline__ uint32_t def_hash(const uint8_t *p, uint32_t hash_bits) {
  return (def_ld32(p) * 2654435761u) >> (32u - hash_bits);
}

// the stream's bits v (n <= 28) at stream bit `at`, OR-ed into the zeroed slot
__device__ __forceinline__ void def_put(uint32_t *sw, uint32_t at, uint32_t v, uint32_t n) {
  if (!n) return;
  const uint32_t b = at + 16u, w = b >> 5;
  const unsigned long long x = (unsigned long long)v << (b & 31u);
  if (w + 1u >= DEF_SLOT_WORDS) return;  // never taken: the block type was chosen to fit (the size check reports it)
  atomicOr(sw + w, (uint32_t)x);
  if ((uint32_t)(x >> 32)) atomicOr(sw + w + 1, (uint32_t)(x >> 32));
}

// scratch of the code builder and the block header, in the hash table's memory between the two passes
struct DeflateScratch {
  uint32_t w[2 * DEF_NLIT];          // weights of the Huffman tree's nodes (leaves first, by weight)
  unsigned short par[2 * DEF_NLIT];  // parent of each node, then its depth
  unsigned short sorted[DEF_NLIT];   // used symbols by (frequency, symbol)
  unsigned short seq[DEF_NLIT + DEF_NDIST];  // the run-length coded code lengths: symbol | extra value << 8
  uint32_t pfreq[DEF_NPRE];
  uint8_t plen[DEF_NPRE];
  unsigned short pcode[DEF_NPRE];
  uint32_t n_seq, hlit, hdist, hclen, btype, bits;
};
// bytes of dynamic shared memory of bvcf_deflate_dyn_kernel at a level: the table, which also holds the scratch
__host__ __device__ constexpr uint32_t def_dyn_smem(const DeflateLevel lv) {
  return ((uint32_t)lv.cands << lv.hash_bits) * 2u > (uint32_t)sizeof(DeflateScratch)
             ? ((uint32_t)lv.cands << lv.hash_bits) * 2u
             : ((uint32_t)sizeof(DeflateScratch) + 15u) & ~15u;
}
static_assert(def_dyn_smem(DEF_LEVELS[9]) <= 48u * 1024u, "no opt-in to more dynamic shared memory");

// lengths of a canonical Huffman code for freq[0 .. n), none longer than maxbits (whole warp).  Unused symbols get 0.  At
// least two symbols get a code (symbols 0 / 1 stand in), as zlib's deflate does, so the code is always complete.  Tree:
// two queues over the leaves ranked by (frequency, symbol); overlong codes: the Kraft-sum repair of miniz
// (tdefl_huffman_enforce_max_code_size), lengths given out by rank, the shortest to the most frequent.
__device__ void def_huff_lengths(const uint32_t *freq, uint32_t n, uint32_t maxbits, uint8_t *len_out, DeflateScratch &s,
                                 int lane) {
  uint32_t m = 0;
  for (uint32_t i0 = 0; i0 < n; i0 += 32) m += __popc(__ballot_sync(FULL, i0 + lane < n && freq[i0 + lane] != 0));
  const bool add0 = m < 2 && freq[0] == 0, add1 = m + (add0 ? 1u : 0u) < 2 && freq[1] == 0;
  m += (add0 ? 1u : 0u) + (add1 ? 1u : 0u);
  auto eff = [&](uint32_t i) -> uint32_t { return (i == 0 && add0) || (i == 1 && add1) ? 1u : freq[i]; };
  for (uint32_t i = lane; i < n; i += 32) {
    len_out[i] = 0;
    const uint32_t fi = eff(i);
    if (!fi) continue;
    uint32_t r = 0;
    for (uint32_t j = 0; j < n; j++) {
      const uint32_t fj = eff(j);
      r += (fj && (fj < fi || (fj == fi && j < i))) ? 1u : 0u;
    }
    s.sorted[r] = (unsigned short)i;
  }
  __syncwarp();
  if (lane == 0) {
    for (uint32_t r = 0; r < m; r++) s.w[r] = eff(s.sorted[r]);
    uint32_t i = 0, j = m;
    for (uint32_t k = m; k < 2 * m - 1; k++) {
      const uint32_t a = (i < m && (j >= k || s.w[i] <= s.w[j])) ? i++ : j++;
      const uint32_t b = (i < m && (j >= k || s.w[i] <= s.w[j])) ? i++ : j++;
      s.w[k] = s.w[a] + s.w[b];
      s.par[a] = s.par[b] = (unsigned short)k;
    }
    s.par[2 * m - 2] = 0;  // the root's depth; a node's parent comes after it, so its depth is known before the node's
    for (int k = (int)(2 * m) - 3; k >= 0; k--) s.par[k] = (unsigned short)(s.par[s.par[k]] + 1u);
    uint32_t cnt[16];
    for (int b = 0; b < 16; b++) cnt[b] = 0;
    for (uint32_t r = 0; r < m; r++) cnt[s.par[r] < maxbits ? s.par[r] : maxbits]++;
    uint32_t total = 0;
    for (uint32_t b = 1; b <= maxbits; b++) total += cnt[b] << (maxbits - b);
    while (total != (1u << maxbits)) {
      cnt[maxbits]--;
      for (uint32_t b = maxbits - 1; b > 0; b--)
        if (cnt[b]) { cnt[b]--; cnt[b + 1] += 2; break; }
      total--;
    }
    uint32_t r = m;
    for (uint32_t b = 1; b <= maxbits; b++)
      for (uint32_t c = cnt[b]; c; c--) len_out[s.sorted[--r]] = (uint8_t)b;
  }
  __syncwarp();
}

// canonical codes (RFC 1951 3.2.2), bit-reversed for the LSB-first stream (one lane)
__device__ void def_canon_codes(const uint8_t *len, uint32_t n, unsigned short *code) {
  uint32_t cnt[16], next[16];
  for (int b = 0; b < 16; b++) cnt[b] = 0;
  for (uint32_t i = 0; i < n; i++) cnt[len[i]]++;
  cnt[0] = 0;
  uint32_t c = 0;
  for (int b = 1; b < 16; b++) { c = (c + cnt[b - 1]) << 1; next[b] = c; }
  for (uint32_t i = 0; i < n; i++)
    code[i] = len[i] ? (unsigned short)(__brev(next[len[i]]++) >> (32 - len[i])) : (unsigned short)0;
}

// One LZ77 pass over the slice.  Every position is hashed and inserted; the positions of a step with the same hash go
// in lane order (grouped with __match_any_sync), and a lane also tries the earlier lanes of its group, so the result is
// what a sequential insertion gives, independent of scheduling.  Positions already covered by a match are not searched.
// HIST: count the tokens' symbols.  Otherwise: emit their codes after `bitpos`, return the end.
template <bool HIST>
__device__ __forceinline__ uint32_t def_lz_pass(const uint8_t *in, uint32_t len, const DeflateLevel lv, unsigned short *tab,
                                                uint32_t *lfreq, uint32_t *dfreq, const unsigned short *lcode,
                                                const uint8_t *llen, const unsigned short *dcode, const uint8_t *dlen,
                                                uint32_t *sw, uint32_t bitpos, int lane) {
  const int k = lv.cands;
  for (uint32_t i = lane; i < (k << lv.hash_bits); i += 32) tab[i] = 0;
  __syncwarp();
  const uint32_t lt = (1u << lane) - 1u;
  uint32_t cur = 0;  // first position not covered by a token yet
  for (uint32_t base = 0; base < len; base += 32) {
    const uint32_t pos = base + (uint32_t)lane;
    const bool hashed = pos + 4u <= len;
    const uint32_t h = hashed ? def_hash(in + pos, lv.hash_bits) : 0xFFFFFFFFu;
    const uint32_t grp = __match_any_sync(FULL, h);
    uint32_t mlen = 0, mdist = 0;
    if (hashed && pos >= cur) def_longest(in, len, pos, base, grp & lt, tab + h * k, k, mlen, mdist);
    __syncwarp();
    if (hashed && lane == __ffs(grp) - 1) {  // the group's first lane puts the group at the front of the row
      unsigned short *row = tab + h * k;
      const int g = __popc(grp);
      for (int j = k - 1; j >= g; j--) row[j] = row[j - g];
      uint32_t mm = grp;
      for (int j = 0; j < g && j < k; j++) {
        const uint32_t l = 31u - __clz(mm);
        mm ^= 1u << l;
        row[j] = (unsigned short)(base + l + 1u);  // slices are 48 KiB: positions + 1 fit 16 bits
      }
    }
    __syncwarp();
    // the parse, in position order: the first lane at or after `c` with a match takes it (lazily: while the next
    // position has a longer one, this one is a literal), the lanes before it are literals
    const uint32_t n_here = len - base < 32u ? len - base : 32u;
    uint32_t c = cur > base ? cur - base : 0u;
    uint32_t role = 0;  // 0 covered, 1 literal, 2 match
    while (c < n_here) {
      const uint32_t mm = __ballot_sync(FULL, mlen != 0 && (uint32_t)lane >= c && (uint32_t)lane < n_here);
      uint32_t f = mm ? (uint32_t)(__ffs(mm) - 1) : n_here;
      if (lv.lazy) {
        while (f < n_here) {
          const uint32_t lf = __shfl_sync(FULL, mlen, (int)f);
          uint32_t ln = 0;
          if (f + 1u < n_here) ln = __shfl_sync(FULL, mlen, (int)f + 1);
          else if (f == 31u && base + 32u + 4u <= len) {  // the next position is the next step's first: search it here
            uint32_t la = 0, ld;                             // (the table holds this step now, as it will then)
            if (lane == 0) {
              const uint32_t p2 = base + 32u, h2 = def_hash(in + p2, lv.hash_bits);
              def_longest(in, len, p2, base, 0u, tab + h2 * k, k, la, ld);
            }
            ln = __shfl_sync(FULL, la, 0);
          }
          if (ln <= lf) break;
          f++;
        }
      }
      if ((uint32_t)lane >= c && (uint32_t)lane < f) role = 1;
      if (f >= n_here) { c = n_here; break; }
      if ((uint32_t)lane == f) role = 2;
      c = f + __shfl_sync(FULL, mlen, (int)f);
    }
    cur = base + c;
    uint32_t ls = 0, le = 0, lev = 0, ds = 0, de = 0, dev = 0;
    if (role == 1) ls = in[pos];
    else if (role == 2) {
      ls = 257u + def_len_sym(mlen, lev, le);
      ds = def_dist_sym(mdist, dev, de);
    }
    if (HIST) {
      if (role) atomicAdd(lfreq + ls, 1u);
      if (role == 2) atomicAdd(dfreq + ds, 1u);
    } else {
      uint32_t na = 0, va = 0, nd = 0, vd = 0;
      if (role) { na = llen[ls] + le; va = (uint32_t)lcode[ls] | (lev << llen[ls]); }
      if (role == 2) { nd = dlen[ds] + de; vd = (uint32_t)dcode[ds] | (dev << dlen[ds]); }
      const uint32_t incl = warp_incl_scan(na + nd, lane);
      const uint32_t at = bitpos + incl - na - nd;
      def_put(sw, at, va, na);
      def_put(sw, at + na, vd, nd);
      bitpos += __shfl_sync(FULL, incl, 31);
    }
  }
  return bitpos;
}

// OR one byte into the slot through its word view (the words around it may be taking reductions of this warp)
__device__ __forceinline__ void def_or_byte(uint8_t *slot, uint32_t i, uint32_t byte) {
  uint32_t *qw = reinterpret_cast<uint32_t *>(slot + (i & ~3u));
  atomicOr(qw, byte << (8u * (i & 3u)));
}

// A slice at levels 2..9: the LZ77 pass runs twice with the same result -- once to count the symbols, once to emit
// them -- so that no token stream is stored.  Between the passes the codes are built from the counts, and the block
// type with the fewest bits is taken: dynamic codes, fixed codes, or a stored block (incompressible text: the member
// is then 18 + 5 + len + 8 bytes, and never more).
__global__ void __launch_bounds__(32) bvcf_deflate_dyn_kernel(const DeflateParams p, const DeflateLevel lv) {
  extern __shared__ __align__(16) unsigned short s_tab[];  // def_dyn_smem(lv) bytes
  __shared__ uint32_t s_crc[256];
  __shared__ uint32_t s_lfreq[DEF_NLIT], s_dfreq[DEF_NDIST];
  __shared__ unsigned short s_lcode[DEF_NLIT], s_dcode[DEF_NDIST];
  __shared__ uint8_t s_llen[DEF_NLIT], s_dlen[DEF_NDIST];
  const int lane = threadIdx.x;
  const uint32_t bi = blockIdx.x;
  if (bi >= p.n_blocks) return;
  const unsigned long long t0 = (unsigned long long)bi * DEF_SLICE;
  const uint32_t len = (uint32_t)(p.text_len - t0 < DEF_SLICE ? p.text_len - t0 : DEF_SLICE);
  const uint8_t *in = p.text + t0;
  uint8_t *slot = p.slots + (size_t)bi * DEF_SLOT;
  uint32_t *sw = reinterpret_cast<uint32_t *>(slot + 16);  // stream bit b is bit (b + 16) % 32 of word (b + 16) / 32
  DeflateScratch &s = *reinterpret_cast<DeflateScratch *>(s_tab);
  for (uint32_t i = lane; i < DEF_NLIT; i += 32) s_lfreq[i] = 0;
  if (lane < (int)DEF_NDIST) s_dfreq[lane] = 0;
  crc_table_init(s_crc, lane);
  __syncwarp();
  const uint32_t crc = crc_warp([&](uint32_t i) { return (uint32_t)in[i]; }, len, lane, s_crc);

  def_lz_pass<true>(in, len, lv, s_tab, s_lfreq, s_dfreq, nullptr, nullptr, nullptr, nullptr, sw, 0, lane);
  if (lane == 0) s_lfreq[256] = 1;  // end of block
  __syncwarp();

  // ---- codes, header, costs ----
  def_huff_lengths(s_lfreq, DEF_NLIT, 15, s_llen, s, lane);
  def_huff_lengths(s_dfreq, DEF_NDIST, 15, s_dlen, s, lane);
  if (lane == 0) {
    uint32_t hlit = DEF_NLIT, hdist = DEF_NDIST;
    while (hlit > 257 && !s_llen[hlit - 1]) hlit--;
    while (hdist > 1 && !s_dlen[hdist - 1]) hdist--;
    // run-length code the hlit + hdist lengths (16: repeat the previous 3-6 times, 17: 3-10 zeros, 18: 11-138 zeros)
    for (int i = 0; i < (int)DEF_NPRE; i++) s.pfreq[i] = 0;
    const uint32_t n = hlit + hdist;
    auto L = [&](uint32_t i) -> uint32_t { return i < hlit ? s_llen[i] : s_dlen[i - hlit]; };
    uint32_t ns = 0;
    auto put = [&](uint32_t sym, uint32_t x) { s.seq[ns++] = (unsigned short)(sym | (x << 8)); s.pfreq[sym]++; };
    for (uint32_t i = 0; i < n;) {
      const uint32_t l = L(i);
      uint32_t run = 1;
      while (i + run < n && L(i + run) == l) run++;
      i += run;
      if (l == 0) {
        while (run >= 11) { const uint32_t r = run < 138 ? run : 138; put(18, r - 11); run -= r; }
        if (run >= 3) { put(17, run - 3); run = 0; }
      } else {
        put(l, 0); run--;
        while (run >= 3) { const uint32_t r = run < 6 ? run : 6; put(16, r - 3); run -= r; }
      }
      for (; run; run--) put(l, 0);
    }
    s.n_seq = ns; s.hlit = hlit; s.hdist = hdist;
  }
  __syncwarp();
  def_huff_lengths(s.pfreq, DEF_NPRE, 7, s.plen, s, lane);
  if (lane == 0) {
    const uint8_t order[DEF_NPRE] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
    uint32_t hclen = DEF_NPRE;
    while (hclen > 4 && !s.plen[order[hclen - 1]]) hclen--;
    unsigned long long dyn = 3 + 5 + 5 + 4 + 3 * hclen, fix = 3;
    for (uint32_t i = 0; i < s.n_seq; i++) {
      const uint32_t sym = s.seq[i] & 0xFFu;
      dyn += s.plen[sym] + (sym == 16 ? 2 : sym == 17 ? 3 : sym == 18 ? 7 : 0);
    }
    for (uint32_t i = 0; i < DEF_NLIT; i++) {
      const unsigned long long f = s_lfreq[i], e = i >= 257 ? def_len_extra(i - 257) : 0;
      dyn += f * (s_llen[i] + e);
      fix += f * (def_fixed_llen(i) + e);
    }
    for (uint32_t d = 0; d < DEF_NDIST; d++) {
      const unsigned long long f = s_dfreq[d];
      dyn += f * (s_dlen[d] + def_dist_extra(d));
      fix += f * (5 + def_dist_extra(d));
    }
    const unsigned long long stored = 8ull * (5 + len);
    const unsigned long long db = (dyn + 7) / 8 * 8, fb = (fix + 7) / 8 * 8;
    s.btype = db <= fb && db <= stored ? 2u : fb <= stored ? 1u : 0u;
    s.bits = (uint32_t)(s.btype == 2 ? dyn : s.btype == 1 ? fix : stored);
    s.hclen = hclen;
    if (s.btype == 1) {
      for (uint32_t i = 0; i < DEF_NLIT; i++) s_llen[i] = (uint8_t)def_fixed_llen(i);
      for (uint32_t d = 0; d < DEF_NDIST; d++) s_dlen[d] = 5;
    }
    if (s.btype) {
      def_canon_codes(s_llen, DEF_NLIT, s_lcode);
      def_canon_codes(s_dlen, DEF_NDIST, s_dcode);
    }
    // the block header: BFINAL = 1, then BTYPE
    if (s.btype == 2) {
      def_canon_codes(s.plen, DEF_NPRE, s.pcode);
      uint32_t bp = 0;
      auto put = [&](uint32_t v, uint32_t nb) { def_put(sw, bp, v, nb); bp += nb; };
      put(1u | (2u << 1), 3);
      put(s.hlit - 257, 5); put(s.hdist - 1, 5); put(hclen - 4, 4);
      for (uint32_t i = 0; i < hclen; i++) put(s.plen[order[i]], 3);
      for (uint32_t i = 0; i < s.n_seq; i++) {
        const uint32_t sym = s.seq[i] & 0xFFu, x = s.seq[i] >> 8;
        put(s.pcode[sym], s.plen[sym]);
        if (sym >= 16) put(x, sym == 16 ? 2 : sym == 17 ? 3 : 7);
      }
    } else if (s.btype == 1) {
      def_put(sw, 0, 1u | (1u << 1), 3);
    }
  }
  __syncwarp();
  const uint32_t btype = s.btype, want = s.bits;
  uint32_t dbytes;
  bool ok = true;
  if (btype == 0) {  // stored: header byte (BFINAL = 1, BTYPE = 00), LEN, NLEN, the text
    uint8_t *d = slot + 18;
    if (lane == 0) {
      d[0] = 1; d[1] = (uint8_t)len; d[2] = (uint8_t)(len >> 8); d[3] = (uint8_t)~len; d[4] = (uint8_t)(~len >> 8);
    }
    for (uint32_t i = lane; i < len; i += 32) d[5 + i] = in[i];
    dbytes = 5 + len;
  } else {
    // the header's bits (dynamic) or 3 (fixed) come first; the header lives in the scratch, which the pass reuses
    uint32_t bitpos = 3;
    if (btype == 2) {
      bitpos = 3 + 5 + 5 + 4 + 3 * s.hclen;
      for (uint32_t i = 0; i < s.n_seq; i++) {
        const uint32_t sym = s.seq[i] & 0xFFu;
        bitpos += s.plen[sym] + (sym == 16 ? 2 : sym == 17 ? 3 : sym == 18 ? 7 : 0);
      }
    }
    __syncwarp();
    bitpos = def_lz_pass<false>(in, len, lv, s_tab, nullptr, nullptr, s_lcode, s_llen, s_dcode, s_dlen, sw, bitpos, lane);
    if (lane == 0) def_put(sw, bitpos, s_lcode[256], s_llen[256]);
    bitpos += s_llen[256];
    ok = bitpos == want;
    dbytes = (bitpos + 7u) >> 3;
  }
  const uint32_t total = 18u + dbytes + 8u;
  __syncwarp();
  __threadfence_block();
  if (lane == 0) {
    const uint8_t hdr[16] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 'B', 'C', 2, 0};
    for (int i = 0; i < 16; i++) slot[i] = hdr[i];
    atomicOr(sw, (total - 1u) & 0xFFFFu);  // BSIZE - 1 (bytes 16, 17 share a word with the first stream bits)
    const uint32_t tr[2] = {crc, len};
    for (uint32_t k = 0; k < 8; k++) def_or_byte(slot, 18u + dbytes + k, (tr[k >> 2] >> (8 * (k & 3))) & 0xFFu);
    p.sizes[bi] = ok ? total : 0u;  // 0: the emitted bits disagree with the counted ones (the host reports it)
  }
}

// blocks of known size back to back: block b goes to out + offs[b] (offs = exclusive prefix of sizes, computed on the host
// side of the call from the sizes it reads back anyway)
struct DeflatePackParams {
  const uint8_t *slots;
  const uint32_t *sizes;
  const unsigned long long *offs;
  uint8_t *out;
  uint32_t n_blocks;
};
__global__ void __launch_bounds__(128) bvcf_deflate_pack_kernel(const DeflatePackParams p) {
  const uint32_t bi = blockIdx.x;
  if (bi >= p.n_blocks) return;
  const uint8_t *src = p.slots + (size_t)bi * DEF_SLOT;
  uint8_t *dst = p.out + p.offs[bi];
  const uint32_t n = p.sizes[bi];
  for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) dst[i] = src[i];
}

}  // namespace bvcf
