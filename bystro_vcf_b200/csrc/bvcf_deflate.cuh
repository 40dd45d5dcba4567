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
// This is a throughput-first compressor (single candidate per hash, no lazy matching, fixed codes): sample-name lists
// deflate about 2.3x with it where `gzip -6` reaches 3-4x.
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
