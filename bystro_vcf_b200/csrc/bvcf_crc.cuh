// bvcf_crc.cuh -- CRC-32 (gzip's, reflected polynomial 0xEDB88320) of text a warp holds, for the deflate kernel (the
// trailer of every block it writes) and the inflate kernel (the check of every member it reads).
//
// A warp computes the CRC of n bytes in one pass: lane l takes a run of them with the byte table, and the runs are joined
// with crc(A || B) = crc(A) * x^(8 |B|) + crc(B) mod P (the identity zlib's crc32_combine uses).  x^(8n) is a product of
// the table entries x^(8 * 2^k) of n's set bits.
#pragma once
#include "bvcf_common.cuh"

namespace bvcf {

__device__ __forceinline__ uint32_t crc_multmodp(uint32_t a, uint32_t b) {  // a * b mod P, reflected CRC-32 polynomial
  uint32_t m = 1u << 31, p = 0;
  for (;;) {
    if (a & m) {
      p ^= b;
      if ((a & (m - 1)) == 0) break;
    }
    m >>= 1;
    b = (b & 1u) ? (b >> 1) ^ 0xEDB88320u : b >> 1;
  }
  return p;
}

// x^(8 * 2^k) mod P, reflected (x^0 is 0x80000000)
__device__ const uint32_t CRC_X8_POW2[32] = {
    0x00800000u, 0x00008000u, 0xedb88320u, 0xb1e6b092u, 0xa06a2517u, 0xed627daeu, 0x88d14467u, 0xd7bbfe6au,
    0xec447f11u, 0x8e7ea170u, 0x6427800eu, 0x4d47bae0u, 0x09fe548fu, 0x83852d0fu, 0x30362f1au, 0x7b5a9cc3u,
    0x31fec169u, 0x9fec022au, 0x6c8dedc4u, 0x15d6874du, 0x5fde7a4eu, 0xbad90e37u, 0x2e4e5eefu, 0x4eaba214u,
    0xa8a472c0u, 0x429a969eu, 0x148d302au, 0xc40ba6d0u, 0xc4e22c3cu, 0x40000000u, 0x20000000u, 0x08000000u};

// crc * x^(8n) mod P: the CRC of the bytes behind `crc` once n more bytes follow them (to be XOR-ed with those bytes' CRC)
__device__ __forceinline__ uint32_t crc_shift(uint32_t crc, uint32_t n) {
  if (n == 0 || crc == 0) return crc;
  uint32_t f = 0x80000000u;
  for (int k = 0; n; n >>= 1, k++)
    if (n & 1u) f = crc_multmodp(CRC_X8_POW2[k], f);
  return crc_multmodp(f, crc);
}

// the byte table, built by the 32 lanes of a warp (__syncwarp before use)
__device__ __forceinline__ void crc_table_init(uint32_t *tab, int lane) {
  for (int i = lane; i < 256; i += 32) {
    uint32_t c = (uint32_t)i;
    for (int k = 0; k < 8; k++) c = (c & 1u) ? (c >> 1) ^ 0xEDB88320u : c >> 1;
    tab[i] = c;
  }
}

// CRC-32 of bytes byte_at(0 .. n), every lane of the warp gets it.  A lane's run is an odd number of 4-byte words, so
// that the 32 lanes read from 32 different shared-memory banks when the bytes are in shared memory.
template <class ByteAt>
__device__ __forceinline__ uint32_t crc_warp(ByteAt byte_at, uint32_t n, int lane, const uint32_t *tab) {
  uint32_t run = ((n + 31u) / 32u + 3u) & ~3u;
  if (((run >> 2) & 1u) == 0) run += 4u;
  const uint32_t lo = (uint32_t)lane * run < n ? (uint32_t)lane * run : n, hi = lo + run < n ? lo + run : n;
  uint32_t c = 0xFFFFFFFFu;
  for (uint32_t i = lo; i < hi; i++) c = tab[(c ^ byte_at(i)) & 0xFFu] ^ (c >> 8);
  c = hi > lo ? crc_shift(c ^ 0xFFFFFFFFu, n - hi) : 0u;  // 0 for an empty run
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) c ^= __shfl_xor_sync(FULL, c, d);
  return c;
}

}  // namespace bvcf
