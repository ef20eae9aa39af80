// dan_zlib.cuh — what the inflate (dan_inflate.cu) and deflate (dan_deflate.cu) kernels share: the DEFLATE (RFC 1951) length / distance
// base and extra-bit tables, the code-length code order, the chunked Adler-32 (RFC 1950) and the chunked CRC-32 (RFC 1952) of a buffer.
#pragma once
#include <cstdint>

constexpr uint32_t kAdlerMod = 65521;

static __constant__ uint16_t kLenBase[29] = {3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258};
static __constant__ uint8_t kLenExtra[29] = {0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0};
static __constant__ uint16_t kDistBase[30] = {1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097,
                                              6145, 8193, 12289, 16385, 24577};
static __constant__ uint8_t kDistExtra[30] = {0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13};
static __constant__ uint8_t kClOrder[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};

// Adler-32 of data[0, total) in independent chunks. Chunk [s, s + m) contributes a = S1 = sum b_k to A and
// b = (total - s) S1 - sum k b_k to B (k local to the chunk), both mod 65521; the parts of any split add up (adler_value).
struct AdlerPart {
  uint64_t a, b;
};

__device__ inline AdlerPart adler_chunk(const uint8_t* data, uint64_t total, uint64_t s, uint64_t m) {
  uint64_t s1 = 0, s2 = 0;
  for (uint64_t k = 0; k < m; ++k) {
    const uint32_t x = data[s + k];
    s1 += x; s2 += (k % kAdlerMod) * x;
    if ((k & 4095) == 4095) { s1 %= kAdlerMod; s2 %= kAdlerMod; }
  }
  s1 %= kAdlerMod; s2 %= kAdlerMod;
  return {s1, ((total - s) % kAdlerMod * s1 + kAdlerMod - s2) % kAdlerMod};
}

// the Adler-32 of data[0, total) from the summed parts of its chunks (each sum below 2^64)
__device__ inline uint32_t adler_value(uint64_t a_sum, uint64_t b_sum, uint64_t total) {
  const uint32_t A = (uint32_t)((1 + a_sum) % kAdlerMod), B = (uint32_t)((total % kAdlerMod + b_sum) % kAdlerMod);
  return (B << 16) | A;
}

// CRC-32 (IEEE 802.3, reflected, as gzip and zlib.crc32) of data[0, total) in independent chunks: each chunk's own CRC (crc32_chunk),
// then, in a fixed order, crc(A B) = crc(A) * x^(8 |B|) mod P ^ crc(B) (crc32_combine, zlib's crc32_combine).
constexpr uint32_t kCrcPoly = 0xedb88320u;

__device__ inline uint32_t crc32_chunk(const uint8_t* data, uint64_t s, uint64_t m) {
  uint32_t c = 0xffffffffu;
  for (uint64_t k = 0; k < m; ++k) {
    c ^= data[s + k];
#pragma unroll
    for (int j = 0; j < 8; ++j) c = (c >> 1) ^ (kCrcPoly & (0u - (c & 1u)));
  }
  return ~c;
}

// a * b modulo P, in the reflected representation (bit 31 is x^0)
__device__ inline uint32_t crc32_multmodp(uint32_t a, uint32_t b) {
  uint32_t p = 0;
  for (uint32_t m = 1u << 31; m; m >>= 1) {
    if (a & m) { p ^= b; if (!(a & (m - 1))) break; }
    b = (b & 1u) ? (b >> 1) ^ kCrcPoly : b >> 1;
  }
  return p;
}

// the CRC-32 of A followed by B from crc_a, crc_b and the length of B
__device__ inline uint32_t crc32_combine(uint32_t crc_a, uint32_t crc_b, uint64_t len_b) {
  uint32_t p = 1u << 31, sq = 1u << 23;                // x^0 and x^8
  for (; len_b; len_b >>= 1) {                         // p = x^(8 len_b) by square-and-multiply
    if (len_b & 1) p = crc32_multmodp(sq, p);
    if (len_b > 1) sq = crc32_multmodp(sq, sq);
  }
  return crc32_multmodp(p, crc_a) ^ crc_b;
}
