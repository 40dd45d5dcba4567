// bvcf_inflate.cuh -- SURVEY 8f-3: bgzf / DEFLATE (RFC 1951) decompression on the GPU, so that the COMPRESSED bytes
// cross PCIe (a 1000 Genomes GT block deflates some 30-50x) and the uncompressed VCF text only ever exists in HBM,
// where the scan kernel reads it.  Upstream of main.go:192 the reference relies on `pigz -d -c` (README.md:10,46:
// "runs at pigz -p 1 limit").
//
// bgzf (the block gzip of bgzip / htslib, what .vcf.gz files are) cuts the stream into independent gzip members of
// at most 64 KiB of text, each with its compressed size in the header: the host walks the headers (a few bytes per
// block), the device inflates the blocks in parallel, ONE WARP PER BLOCK.  Inside a block DEFLATE is serial (Huffman
// codes of unknown length, matches that copy from the bytes just written), so:
//   * every lane runs the same bit reader and the same canonical Huffman decode (count / symbol arrays in shared
//     memory, code length by code length as in zlib's puff.c): uniform control flow, no broadcasts;
//   * the block's text is built in shared memory (a 16 KiB ring per warp), where a match is a PARALLEL copy -- lane i writes
//     byte i, reading byte (i mod distance) of the source, so even the distance-4 runs of genotype text ("0|0\t"
//     repeated 64 times per match) move 32 bytes per step instead of waiting on a store-to-load round trip per byte;
//   * the finished block leaves as coalesced 16-byte stores.
// Stored, fixed and dynamic blocks are all handled.  Every member is checked against its gzip trailer: ISIZE, and the
// CRC-32 of the text, computed from the shared-memory ring as each piece is flushed (bvcf_crc.cuh), so the check makes
// no second pass over the text in HBM.  The bit reader is bounded: a stream that would consume more bits than its
// payload holds (a chain of empty blocks, a missing end-of-block code, a truncated payload) fails its block, and no
// read goes further than 11 bytes past the payload.
// (A first version gave a THREAD per block with its text in global memory: 12 GB/s -- every byte of an overlapping
// match waited for the previous store to come back from L2.)
#pragma once
#include "bvcf_common.cuh"
#include "bvcf_crc.cuh"

namespace bvcf {

struct InflateBlock {
  unsigned long long in_off;   // first byte of the block's DEFLATE payload in `comp`
  unsigned long long out_off;  // where its text goes in `out`
  uint32_t in_len;             // payload bytes
  uint32_t out_len;            // ISIZE: bytes of text
  uint32_t crc;                // CRC-32 of the text (the gzip trailer)
  uint32_t pad;
};
struct InflateParams {
  const uint8_t *comp;
  uint8_t *out;
  const InflateBlock *blocks;
  uint32_t n_blocks;
  uint32_t *n_bad;             // blocks that failed (corrupt stream, size or CRC-32 mismatch)
};

constexpr int INF_MAXBITS = 15, INF_MAXL = 288, INF_MAXD = 30;

struct InfBits {
  const uint8_t *p;            // next input byte
  const uint8_t *end;
  unsigned long long buf;      // bits not yet consumed, LSB first
  int cnt;
  __device__ __forceinline__ void refill() {  // at least 32 bits afterwards
    if (cnt <= 32) {
      // four bytes at any alignment from two aligned words; just past `end` lie the member's trailer and the next
      // block's header (or the buffer's slack): harmless, a valid stream stops at its end-of-block symbol.  Further out
      // nothing is read -- zeros come in, and overrun() fails the block at its next check
      uint32_t w = 0;
      if (p <= end + 4) {
        const uint32_t *wp = reinterpret_cast<const uint32_t *>((uintptr_t)p & ~(uintptr_t)3);
        const uint32_t sh = (uint32_t)((uintptr_t)p & 3u) * 8u;
        w = __funnelshift_r(wp[0], wp[1], sh);
      }
      buf |= (unsigned long long)w << cnt;
      cnt += 32;
      p += 4;
    }
  }
  __device__ __forceinline__ uint32_t bits(int n) {  // n <= 32
    if (cnt < n) refill();
    const uint32_t v = (uint32_t)(buf & ((1ull << n) - 1ull));
    buf >>= n; cnt -= n;
    return v;
  }
  // more bits consumed than the payload holds
  __device__ __forceinline__ bool overrun() const { return (long long)(p - end) * 8 > (long long)cnt; }
};

struct InfHuff {
  short *count;          // [INF_MAXBITS + 1] codes of each length
  short *symbol;         // symbols ordered by code
  unsigned short *lut;   // (1 << lut_bits) entries: symbol << 4 | code length for codes of at most lut_bits bits, else 0xFFFF
  int lut_bits;
};

// Huffman decode: one table lookup for codes of at most lut_bits bits (all but the rarest symbols), else the canonical
// walk, one bit at a time (puff.c)
__device__ __forceinline__ int inf_decode(InfBits &b, const InfHuff &h) {
  if (b.cnt < INF_MAXBITS) b.refill();
  {
    const uint32_t e = h.lut[(uint32_t)b.buf & ((1u << h.lut_bits) - 1u)];
    if (e != 0xFFFFu) {
      const int len = (int)(e & 15u);
      b.buf >>= len; b.cnt -= len;
      return (int)(e >> 4);
    }
  }
  int code = 0, first = 0, index = 0;
  unsigned long long buf = b.buf;
  for (int len = 1; len <= INF_MAXBITS; len++) {
    code |= (int)(buf & 1ull);
    buf >>= 1;
    const int count = h.count[len];
    if (code - count < first) {
      b.buf = buf; b.cnt -= len;
      return h.symbol[index + (code - first)];
    }
    index += count;
    first += count;
    first <<= 1;
    code <<= 1;
  }
  return -1;
}

// count / symbol tables from code lengths; returns < 0 for an over-subscribed set
__device__ __forceinline__ int inf_construct1(InfHuff &h, const short *length, int n) {
  for (int len = 0; len <= INF_MAXBITS; len++) h.count[len] = 0;
  for (int s = 0; s < n; s++) h.count[length[s]]++;
  if (h.count[0] == n) return 0;
  int left = 1;
  for (int len = 1; len <= INF_MAXBITS; len++) {
    left <<= 1;
    left -= h.count[len];
    if (left < 0) return left;
  }
  short offs[INF_MAXBITS + 1];
  offs[1] = 0;
  for (int len = 1; len < INF_MAXBITS; len++) offs[len + 1] = offs[len] + h.count[len];
  for (int s = 0; s < n; s++)
    if (length[s] != 0) h.symbol[offs[length[s]]++] = (short)s;
  return left;
}

// the tables live in shared memory: lane 0 builds them (read-modify-write counters), everyone waits
__device__ __forceinline__ int inf_construct(InfHuff &h, const short *length, int n) {
  __syncwarp();
  int r = 0;
  if ((threadIdx.x & 31) == 0) r = inf_construct1(h, length, n);
  r = __shfl_sync(FULL, r, 0);
  __syncwarp();
  // the lookup table: entry i = the symbol whose bit-reversed code is the low bits of i (DEFLATE sends Huffman codes
  // most significant bit first into a least-significant-bit-first stream)
  const int lane = threadIdx.x & 31, B = h.lut_bits;
  for (int i = lane; i < (1 << B); i += 32) h.lut[i] = 0xFFFFu;
  __syncwarp();
  int used = 0;
  for (int len = 1; len <= INF_MAXBITS; len++) used += h.count[len];
  for (int j = lane; j < used; j += 32) {  // the j-th symbol in code order
    int len = 1, first = 0, index = 0;     // its length and code: walk the counts
    while (j >= index + h.count[len]) { index += h.count[len]; first = (first + h.count[len]) << 1; len++; }
    if (len <= B) {
      const uint32_t code = (uint32_t)(first + (j - index));
      const uint32_t rev = __brev(code) >> (32 - len);
      const unsigned short e = (unsigned short)(((uint32_t)h.symbol[j] << 4) | (uint32_t)len);
      for (uint32_t k = rev; k < (1u << B); k += 1u << len) h.lut[k] = e;
    }
  }
  __syncwarp();
  return r;
}

__device__ const short INF_LBASE[29] = {3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258};
__device__ const short INF_LEXT[29] = {0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0};
__device__ const short INF_DBASE[30] = {1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097, 6145, 8193, 12289, 16385, 24577};
__device__ const short INF_DEXT[30] = {0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13};
__device__ const unsigned char INF_ORDER[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};

// The text of a block goes through a 16 KiB ring in shared memory: text byte t lives at ring byte t & INF_RING_MASK.
// Finished 4 KiB pieces leave for global memory as soon as the decoder is 4 KiB past them -- long before their ring
// bytes are written again.  DEFLATE matches reach back 32 KiB: a source byte that has left the ring (more than
// 16 KiB - 258 behind the decoder, so flushed at least 7 KiB ago) is read back from the text in global memory.  Half the
// ring of the first version: 10 resident warps per SM instead of 7 for a kernel that is one serial chain per warp.
constexpr uint32_t INF_RING = 16384, INF_RING_MASK = INF_RING - 1, INF_PIECE = 4096;
static_assert(2 * INF_PIECE + 258 + 1 < INF_RING - 258, "a byte outside the ring has been flushed");
struct InfOut {
  uint32_t ring_s;     // shared-memory byte address of the ring
  const uint8_t *ring; // the same, generic
  uint8_t *g;          // where text byte 0 goes in global memory
  uint32_t o;          // text bytes produced
  uint32_t flushed;    // text bytes already in global memory (a multiple of INF_PIECE until the end)
  uint32_t out_len;
  uint32_t crc;        // CRC-32 of the flushed text
  const uint32_t *crc_tab;  // its byte table, in shared memory
};
// text bytes [from, to) ring -> global, all lanes; coalesced 4-byte words where the alignment allows.  Their CRC-32 is
// folded into w.crc on the way (the bytes are read from the ring, not from HBM)
__device__ __forceinline__ void inf_flush(InfOut &w, uint32_t from, uint32_t to, int lane) {
  uint8_t *g = w.g;
  uint32_t a = from;
  // bytes up to the first 4-byte boundary of the destination
  const uint32_t head = (4u - (uint32_t)((uintptr_t)(g + a) & 3u)) & 3u;
  const uint32_t h = head < to - a ? head : to - a;
  if ((uint32_t)lane < h) g[a + lane] = w.ring[(a + lane) & INF_RING_MASK];
  a += h;
  const uint32_t nw = (to - a) >> 2;
  for (uint32_t i = lane; i < nw; i += 32) {
    const uint32_t t = a + 4 * i;  // four text bytes, any alignment in the ring
    const uint32_t r0 = t & INF_RING_MASK;
    uint32_t v;
    if ((r0 & 3u) == 0) v = *reinterpret_cast<const uint32_t *>(w.ring + r0);
    else v = (uint32_t)w.ring[r0] | ((uint32_t)w.ring[(t + 1) & INF_RING_MASK] << 8) | ((uint32_t)w.ring[(t + 2) & INF_RING_MASK] << 16) |
             ((uint32_t)w.ring[(t + 3) & INF_RING_MASK] << 24);
    *reinterpret_cast<uint32_t *>(g + t) = v;
  }
  a += 4 * nw;
  if (a + lane < to) g[a + lane] = w.ring[(a + lane) & INF_RING_MASK];
  const uint8_t *ring = w.ring;
  const uint32_t c = crc_warp([&](uint32_t i) { return (uint32_t)ring[(from + i) & INF_RING_MASK]; }, to - from, lane, w.crc_tab);
  w.crc = crc_shift(w.crc, to - from) ^ c;
}

// literal/length + distance codes until the end-of-block symbol; every lane runs this in lockstep; returns 0 or an error
__device__ __forceinline__ int inf_codes(InfBits &b, const InfHuff &lc, const InfHuff &dc, InfOut &w, int lane) {
  for (;;) {
    if (w.o - w.flushed >= 2 * INF_PIECE) {  // a finished piece, 8 KiB behind the decoder: out it goes
      __syncwarp();
      inf_flush(w, w.flushed, w.flushed + INF_PIECE, lane);
      w.flushed += INF_PIECE;
    }
    int sym = inf_decode(b, lc);
    if (sym < 0) return 1;
    if (sym < 256) {
      if (w.o >= w.out_len) return 2;
      if (lane == 0) asm volatile("st.shared.u8 [%0], %1;\n" ::"r"(w.ring_s + (w.o & INF_RING_MASK)), "r"(sym) : "memory");
      w.o++;
    } else if (sym == 256) {
      return b.overrun() ? 18 : 0;
    } else {
      sym -= 257;
      if (sym >= 29) return 3;
      const uint32_t len = (uint32_t)INF_LBASE[sym] + b.bits(INF_LEXT[sym]);
      const int ds = inf_decode(b, dc);
      if (ds < 0 || ds >= 30) return 4;
      const uint32_t dist = (uint32_t)INF_DBASE[ds] + b.bits(INF_DEXT[ds]);
      if (dist > w.o) return 5;           // bgzf blocks are independent: no history before the block
      if (w.o + len > w.out_len) return 2;
      __syncwarp();                       // the literals and matches written so far are visible to every lane
      const uint32_t src = w.o - dist, dst = w.o;
      if (dist >= len) {                  // plain copy
        // text bytes below ring_lo are no longer in the ring (or are about to be overwritten by this very match)
        const uint32_t ring_lo = w.o + len > INF_RING ? w.o + len - INF_RING : 0u;
        if (src >= ring_lo) {
          for (uint32_t i = lane; i < len; i += 32) {
            uint32_t c;
            asm volatile("ld.shared.u8 %0, [%1];\n" : "=r"(c) : "r"(w.ring_s + ((src + i) & INF_RING_MASK)) : "memory");
            asm volatile("st.shared.u8 [%0], %1;\n" ::"r"(w.ring_s + ((dst + i) & INF_RING_MASK)), "r"(c) : "memory");
          }
        } else {                          // a far match: (part of) its source was flushed long ago
          for (uint32_t i = lane; i < len; i += 32) {
            uint32_t c;
            if (src + i >= ring_lo) asm volatile("ld.shared.u8 %0, [%1];\n" : "=r"(c) : "r"(w.ring_s + ((src + i) & INF_RING_MASK)) : "memory");
            else c = __ldcg(w.g + src + i);  // L2: written by this warp's own flush, ordered by the __syncwarp() above
            asm volatile("st.shared.u8 [%0], %1;\n" ::"r"(w.ring_s + ((dst + i) & INF_RING_MASK)), "r"(c) : "memory");
          }
        }
      } else {                            // the source runs into the bytes being written: byte i repeats byte i mod dist
        uint32_t m, step;
        if ((dist & (dist - 1u)) == 0) { m = (uint32_t)lane & (dist - 1u); step = 32u & (dist - 1u); }
        else { m = (uint32_t)lane % dist; step = 32u % dist; }
        for (uint32_t i = lane; i < len; i += 32) {
          uint32_t c;
          asm volatile("ld.shared.u8 %0, [%1];\n" : "=r"(c) : "r"(w.ring_s + ((src + m) & INF_RING_MASK)) : "memory");
          asm volatile("st.shared.u8 [%0], %1;\n" ::"r"(w.ring_s + ((dst + i) & INF_RING_MASK)), "r"(c) : "memory");
          m += step;
          if (m >= dist) m -= dist;
        }
      }
      __syncwarp();
      w.o += len;
    }
  }
}

constexpr uint32_t INF_TEXT_MAX = 65536;  // a bgzf block holds at most 64 KiB of text
constexpr int INF_LBITS = 10, INF_DBITS = 9;  // lookup-table bits of the literal/length and the distance code
constexpr uint32_t INF_TAB_SHORTS = 2 * (INF_MAXBITS + 1) + INF_MAXL + INF_MAXD + 2 + INF_MAXL + INF_MAXD + 2 + 16;
constexpr uint32_t INF_LUT_BYTES = 2 * ((1u << INF_LBITS) + (1u << INF_DBITS));
constexpr uint32_t INF_SMEM = INF_RING + 2 * INF_TAB_SHORTS + INF_LUT_BYTES + 256 * 4;  // ring, code tables, CRC-32 table
static_assert((INF_RING + 2 * INF_TAB_SHORTS + INF_LUT_BYTES) % 4 == 0, "the CRC-32 table is word-aligned");

__global__ void __launch_bounds__(32) bvcf_inflate_kernel(const InflateParams p) {
  extern __shared__ __align__(16) uint8_t s_inf[];
  const int lane = threadIdx.x;
  const uint32_t bi = blockIdx.x;
  if (bi >= p.n_blocks) return;
  const InflateBlock blk = p.blocks[bi];
  short *tabs = reinterpret_cast<short *>(s_inf + INF_RING);
  short *lencnt = tabs, *distcnt = tabs + 16, *lensym = tabs + 32, *distsym = lensym + INF_MAXL, *lengths = distsym + INF_MAXD + 2;
  unsigned short *llut = reinterpret_cast<unsigned short *>(tabs + INF_TAB_SHORTS), *dlut = llut + (1 << INF_LBITS);
  uint32_t *crc_tab = reinterpret_cast<uint32_t *>(s_inf + INF_RING + 2 * INF_TAB_SHORTS + INF_LUT_BYTES);
  crc_table_init(crc_tab, lane);  // ordered before its first use by the __syncwarp() in front of every flush
  int err = blk.out_len > INF_TEXT_MAX ? 17 : 0;
  InfBits b;
  b.p = p.comp + blk.in_off; b.end = b.p + blk.in_len; b.buf = 0; b.cnt = 0;
  InfOut w;
  w.ring_s = (uint32_t)__cvta_generic_to_shared(s_inf); w.ring = s_inf; w.g = p.out + blk.out_off;
  w.o = 0; w.flushed = 0; w.out_len = blk.out_len; w.crc = 0; w.crc_tab = crc_tab;
  InfHuff lc, dc;
  lc.count = lencnt; lc.symbol = lensym; dc.count = distcnt; dc.symbol = distsym;
  lc.lut = llut; lc.lut_bits = INF_LBITS; dc.lut = dlut; dc.lut_bits = INF_DBITS;
  int last = 1;
  if (!err) do {
    if (b.overrun()) { err = 19; break; }  // e.g. a chain of empty blocks running past the payload
    last = (int)b.bits(1);
    const int type = (int)b.bits(2);
    if (type == 0) {  // stored
      b.buf >>= (b.cnt & 7); b.cnt &= ~7;  // to the byte boundary
      // the bit buffer holds whole bytes now: give them back
      b.p -= b.cnt >> 3; b.buf = 0; b.cnt = 0;
      if (b.p + 4 > b.end) { err = 6; break; }
      const uint32_t len = (uint32_t)b.p[0] | ((uint32_t)b.p[1] << 8), nlen = (uint32_t)b.p[2] | ((uint32_t)b.p[3] << 8);
      b.p += 4;
      if ((len ^ 0xFFFFu) != nlen || b.p + len > b.end || w.o + len > blk.out_len) { err = 7; break; }
      // a stored block may be longer than the ring: straight to global memory, and into the ring for later matches
      __syncwarp();
      inf_flush(w, w.flushed, w.o, lane);
      for (uint32_t i = lane; i < len; i += 32) {
        const uint8_t c = b.p[i];
        w.g[w.o + i] = c;
        s_inf[(w.o + i) & INF_RING_MASK] = c;
      }
      const uint8_t *src = b.p;
      const uint32_t c = crc_warp([&](uint32_t i) { return (uint32_t)src[i]; }, len, lane, crc_tab);
      w.crc = crc_shift(w.crc, len) ^ c;
      w.o += len; b.p += len;
      w.flushed = w.o;
      __syncwarp();
    } else if (type == 1) {  // fixed codes
      __syncwarp();
      int s = 0;
      for (; s < 144; s++) lengths[s] = 8;
      for (; s < 256; s++) lengths[s] = 9;
      for (; s < 280; s++) lengths[s] = 7;
      for (; s < 288; s++) lengths[s] = 8;
      inf_construct(lc, lengths, 288);
      for (s = 0; s < 30; s++) lengths[s] = 5;
      inf_construct(dc, lengths, 30);
      err = inf_codes(b, lc, dc, w, lane);
    } else if (type == 2) {  // dynamic codes
      const int nlen = (int)b.bits(5) + 257, ndist = (int)b.bits(5) + 1, ncode = (int)b.bits(4) + 4;
      if (nlen > 286 || ndist > 30) { err = 8; break; }
      __syncwarp();
      int idx = 0;
      for (; idx < ncode; idx++) lengths[INF_ORDER[idx]] = (short)b.bits(3);
      for (; idx < 19; idx++) lengths[INF_ORDER[idx]] = 0;
      if (inf_construct(lc, lengths, 19) != 0) { err = 9; break; }  // the code length code must be complete
      idx = 0;
      while (idx < nlen + ndist) {
        int sym = inf_decode(b, lc);
        if (sym < 0) { err = 10; break; }
        if (sym < 16) {
          lengths[idx++] = (short)sym;
        } else {
          int len = 0, rep;
          if (sym == 16) {
            if (idx == 0) { err = 11; break; }
            len = lengths[idx - 1];
            rep = 3 + (int)b.bits(2);
          } else if (sym == 17) {
            rep = 3 + (int)b.bits(3);
          } else {
            rep = 11 + (int)b.bits(7);
          }
          if (idx + rep > nlen + ndist) { err = 12; break; }
          while (rep--) lengths[idx++] = (short)len;
        }
      }
      if (err) break;
      if (b.overrun()) { err = 20; break; }
      __syncwarp();
      if (lengths[256] == 0) { err = 13; break; }
      // an incomplete code is allowed only as a single code of one bit (RFC 1951 3.2.7, as zlib and puff.c read it)
      int r = inf_construct(lc, lengths, nlen);
      if (r < 0 || (r > 0 && !(lc.count[1] == 1 && nlen - lc.count[0] == 1))) { err = 14; break; }
      r = inf_construct(dc, lengths + nlen, ndist);
      if (r < 0 || (r > 0 && !(dc.count[1] == 1 && ndist - dc.count[0] == 1))) { err = 15; break; }
      err = inf_codes(b, lc, dc, w, lane);
    } else {
      err = 16;
    }
  } while (!last && !err);
  __syncwarp();
  if (err || w.o != blk.out_len) {
    if (lane == 0) atomicAdd(p.n_bad, 1u);
    return;
  }
  inf_flush(w, w.flushed, w.o, lane);  // what is still in the ring
  if (w.crc != blk.crc && lane == 0) atomicAdd(p.n_bad, 1u);
}

}  // namespace bvcf
