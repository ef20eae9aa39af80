// dan_inflate.cu — batched zlib (RFC 1950 / 1951) inflate on the GPU: n independent streams into fixed-size output slots.
//
// One warp per stream, kWarps streams per CTA. Every lane of the warp runs the same bit reader and the same symbol decode (the loads
// are warp-uniform broadcasts), so control flow never diverges and no shuffles are needed to share a symbol; the lanes split the
// byte work: stored blocks and matches are copied 32 bytes a round, and the Adler-32 of the slot is summed over 32 chunks once the
// stream ends. Decode tables of each Huffman block live in the warp's shared memory: a 2^kLitBits / 2^kDistBits first-level lookup
// (symbol | length << 9), with a canonical bit-by-bit decode (puff's count[] / symbol[] arrays) for the rare longer codes.
//
// Every input read is bounds-checked against the stream's [0, len); every output write against the slot; a distance may not reach
// behind the output already produced; over-subscribed and incomplete code-length sets are rejected as zlib rejects them. A stream
// that fails gets its status and an all-zero slot; it never touches another stream's slot or status.
#include <cstdint>
#include <cuda_runtime.h>
#include "dan_internal.h"
#include "dan_zlib.cuh"

namespace {

constexpr int kWarps = 4;                  // streams per CTA
constexpr int kLitBits = 10, kDistBits = 8;
constexpr int kMaxBits = 15;

struct Huff {                              // one decode table set
  uint16_t count[kMaxBits + 1];            // codes of each length
  uint16_t symbol[288];                    // symbols in canonical order
  uint16_t fast[1 << kLitBits];            // first-level lookup: symbol | len << 9, len 0 = longer code or no code
};

struct WarpSmem {
  Huff lit, dist;
  uint8_t lens[288 + 32];                  // code lengths of the current block: literal/length at [0, 288), distance at [288, 320)
  uint8_t cl[19];                          // code-length code lengths of a dynamic block
};

// Warp-uniform LSB-first bit reader over src[0, len).
struct Bits {
  const uint8_t* src;
  uint32_t len, pos;                       // next byte to load
  uint64_t buf;
  int cnt;
  __device__ void refill() {
    while (cnt <= 56 && pos < len) { buf |= (uint64_t)__ldg(src + pos) << cnt; ++pos; cnt += 8; }
  }
  // n <= 32 bits; false when the stream ends first
  __device__ bool take(int n, uint32_t* v) {
    if (cnt < n) { refill(); if (cnt < n) return false; }
    *v = (uint32_t)(buf & ((1ull << n) - 1)); buf >>= n; cnt -= n;
    return true;
  }
};

// Builds `h` from lens[0, n) with all lanes. Returns 0, or -1 for a set zlib rejects: over-subscribed, or incomplete unless it has no
// codes at all or (outside the code-length code) a single one-bit code. `fast_bits` <= kLitBits entries of h.fast are filled.
__device__ int build_huff(Huff& h, const uint8_t* lens, int n, int fast_bits, bool code_length_code, int lane) {
  int rc = 0;
  if (lane == 0) {
    for (int l = 0; l <= kMaxBits; ++l) h.count[l] = 0;
    for (int s = 0; s < n; ++s) h.count[lens[s]]++;
    int max = kMaxBits;
    while (max > 0 && h.count[max] == 0) --max;
    int left = 1;
    for (int l = 1; l <= kMaxBits; ++l) { left <<= 1; left -= h.count[l]; if (left < 0) { rc = -1; break; } }
    if (rc == 0 && max > 0 && left > 0 && (code_length_code || max != 1)) rc = -1;
    if (rc == 0) {
      uint16_t offs[kMaxBits + 1];
      offs[1] = 0;
      for (int l = 1; l < kMaxBits; ++l) offs[l + 1] = offs[l] + h.count[l];
      for (int s = 0; s < n; ++s) if (lens[s]) h.symbol[offs[lens[s]]++] = (uint16_t)s;
    }
  }
  rc = __shfl_sync(0xffffffffu, rc, 0);
  __syncwarp();
  if (rc) return rc;
  // entry e: the next fast_bits input bits, LSB first, decoded canonically
  for (int e = lane; e < (1 << fast_bits); e += 32) {
    int code = 0, first = 0, index = 0;
    uint16_t ent = 0;
    for (int l = 1; l <= fast_bits; ++l) {
      code |= (e >> (l - 1)) & 1;
      const int c = h.count[l];
      if (code - first < c) { ent = (uint16_t)(h.symbol[index + code - first] | (l << 9)); break; }
      index += c; first += c; first <<= 1; code <<= 1;
    }
    h.fast[e] = ent;
  }
  __syncwarp();
  return 0;
}

// one symbol: >= 0, or -1 when the input ends, -2 for a bit pattern that is no code
__device__ int decode_sym(Bits& b, const Huff& h, int fast_bits) {
  if (b.cnt < kMaxBits) b.refill();
  const uint16_t ent = h.fast[b.buf & ((1u << fast_bits) - 1)];
  const int l = ent >> 9;
  if (l) {
    if (l > b.cnt) return -1;
    b.buf >>= l; b.cnt -= l;
    return ent & 511;
  }
  int code = 0, first = 0, index = 0;
  for (int len = 1; len <= kMaxBits; ++len) {
    if (len > b.cnt) return -1;
    code |= (int)((b.buf >> (len - 1)) & 1);
    const int c = h.count[len];
    if (code - first < c) { b.buf >>= len; b.cnt -= len; return h.symbol[index + code - first]; }
    index += c; first += c; first <<= 1; code <<= 1;
  }
  return -2;
}

__global__ void __launch_bounds__(kWarps * 32) inflate_kernel(const uint8_t* __restrict__ src, const uint64_t* __restrict__ offsets,
                                                                const uint32_t* __restrict__ lengths, int n, uint8_t* dst,
                                                                uint64_t slot_bytes, int32_t* __restrict__ status) {
  __shared__ WarpSmem smem[kWarps];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int i = blockIdx.x * kWarps + w;
  if (i >= n) return;
  WarpSmem& sm = smem[w];
  uint8_t* out = dst + (uint64_t)i * slot_bytes;
  Bits b{src + offsets[i], lengths[i], 0, 0, 0};
  uint64_t o = 0;                                     // bytes written
  int st = DAN_INFLATE_OK;
  uint32_t v, v2;
  // zlib header: CM 8, CINFO <= 7, FCHECK, no preset dictionary
  if (!b.take(8, &v) || !b.take(8, &v2)) st = DAN_INFLATE_E_INPUT;
  else if ((v & 15) != 8 || (v >> 4) > 7 || ((v << 8) | v2) % 31 != 0 || (v2 & 0x20)) st = DAN_INFLATE_E_HEADER;
  bool last = false;
  while (st == DAN_INFLATE_OK && !last) {
    uint32_t type;
    if (!b.take(1, &v) || !b.take(2, &type)) { st = DAN_INFLATE_E_INPUT; break; }
    last = v != 0;
    if (type == 0) {                                  // stored: LEN / NLEN at the next byte boundary, then LEN raw bytes
      b.buf >>= b.cnt & 7; b.cnt &= ~7;
      uint32_t ln, nln;
      if (!b.take(16, &ln) || !b.take(16, &nln)) { st = DAN_INFLATE_E_INPUT; break; }
      if (ln != (~nln & 0xffffu)) { st = DAN_INFLATE_E_BLOCK; break; }
      const uint32_t inbuf = b.cnt >> 3;              // whole bytes still in the bit buffer come first
      const uint32_t in_pos = b.pos - inbuf;
      if (ln > b.len - in_pos) { st = DAN_INFLATE_E_INPUT; break; }
      if (ln > slot_bytes - o) { st = DAN_INFLATE_E_OUTPUT_LONG; break; }
      for (uint32_t k = lane; k < ln; k += 32) out[o + k] = __ldg(b.src + in_pos + k);
      o += ln;
      b.pos = in_pos + ln; b.buf = 0; b.cnt = 0;
      continue;
    }
    if (type == 3) { st = DAN_INFLATE_E_BLOCK; break; }
    if (type == 1) {                                  // fixed Huffman codes (RFC 1951 §3.2.6); 32 five-bit distance codes, 30 and 31 unused
      for (int s = lane; s < 288 + 32; s += 32) sm.lens[s] = s < 144 ? 8 : s < 256 ? 9 : s < 280 ? 7 : s < 288 ? 8 : 5;
      __syncwarp();
    } else {                                          // dynamic: HLIT, HDIST, HCLEN, the code-length code, then the run-length coded lengths
      uint32_t hlit, hdist, hclen;
      if (!b.take(5, &hlit) || !b.take(5, &hdist) || !b.take(4, &hclen)) { st = DAN_INFLATE_E_INPUT; break; }
      const int nlen = hlit + 257, ndist = hdist + 1;
      if (nlen > 286 || ndist > 30) { st = DAN_INFLATE_E_CODES; break; }
      bool ok = true;
      for (uint32_t k = 0; k < 19; ++k) {
        uint32_t x = 0;
        if (k < hclen + 4 && !b.take(3, &x)) { ok = false; break; }
        if (lane == 0) sm.cl[kClOrder[k]] = (uint8_t)x;
      }
      if (!ok) { st = DAN_INFLATE_E_INPUT; break; }
      for (int s = lane; s < 288 + 32; s += 32) sm.lens[s] = 0;
      __syncwarp();
      if (build_huff(sm.dist, sm.cl, 19, 7, true, lane)) { st = DAN_INFLATE_E_CODES; break; }     // the distance table is free until below
      // length k of the nlen + ndist: literal/length k at lens[k], distance k - nlen at lens[288 + k - nlen]
      auto at = [&](int k) { return k < nlen ? k : 288 + k - nlen; };
      int k = 0;
      while (k < nlen + ndist) {
        const int sym = decode_sym(b, sm.dist, 7);
        if (sym < 0) { st = sym == -1 ? DAN_INFLATE_E_INPUT : DAN_INFLATE_E_CODES; break; }
        if (sym < 16) { if (lane == 0) sm.lens[at(k)] = (uint8_t)sym; ++k; continue; }
        uint32_t rep; int val = 0;
        if (sym == 16) {
          if (k == 0) { st = DAN_INFLATE_E_CODES; break; }
          __syncwarp();
          val = sm.lens[at(k - 1)];
          if (!b.take(2, &rep)) { st = DAN_INFLATE_E_INPUT; break; }
          rep += 3;
        } else if (sym == 17) {
          if (!b.take(3, &rep)) { st = DAN_INFLATE_E_INPUT; break; }
          rep += 3;
        } else {
          if (!b.take(7, &rep)) { st = DAN_INFLATE_E_INPUT; break; }
          rep += 11;
        }
        if (k + (int)rep > nlen + ndist) { st = DAN_INFLATE_E_CODES; break; }
        if (lane == 0) for (uint32_t r = 0; r < rep; ++r) sm.lens[at(k + (int)r)] = (uint8_t)val;
        k += rep;
      }
      if (st != DAN_INFLATE_OK) break;
      __syncwarp();
      if (sm.lens[256] == 0) { st = DAN_INFLATE_E_CODES; break; }                 // no end-of-block code
    }
    if (build_huff(sm.lit, sm.lens, 288, kLitBits, false, lane) || build_huff(sm.dist, sm.lens + 288, 32, kDistBits, false, lane)) {
      st = DAN_INFLATE_E_CODES; break;
    }
    // symbols of the block
    while (true) {
      const int sym = decode_sym(b, sm.lit, kLitBits);
      if (sym < 0) { st = sym == -1 ? DAN_INFLATE_E_INPUT : DAN_INFLATE_E_CODES; break; }
      if (sym < 256) {
        if (o >= slot_bytes) { st = DAN_INFLATE_E_OUTPUT_LONG; break; }
        if (lane == 0) out[o] = (uint8_t)sym;
        ++o;
        continue;
      }
      if (sym == 256) break;
      const int ls = sym - 257;
      if (ls >= 29) { st = DAN_INFLATE_E_CODES; break; }
      uint32_t e;
      if (!b.take(kLenExtra[ls], &e)) { st = DAN_INFLATE_E_INPUT; break; }
      const uint32_t len = kLenBase[ls] + e;
      const int ds = decode_sym(b, sm.dist, kDistBits);
      if (ds < 0) { st = ds == -1 ? DAN_INFLATE_E_INPUT : DAN_INFLATE_E_CODES; break; }
      if (ds >= 30) { st = DAN_INFLATE_E_CODES; break; }
      if (!b.take(kDistExtra[ds], &e)) { st = DAN_INFLATE_E_INPUT; break; }
      const uint32_t dist = kDistBase[ds] + e;
      if (dist > o) { st = DAN_INFLATE_E_DISTANCE; break; }
      if (len > slot_bytes - o) { st = DAN_INFLATE_E_OUTPUT_LONG; break; }
      __syncwarp();                                   // earlier bytes written by other lanes are visible
      // byte o + j repeats byte o - dist + j % dist: every source byte precedes o, so the rounds need no ordering among themselves
      const uint8_t* from = out + o - dist;
      for (uint32_t j = lane; j < len; j += 32) out[o + j] = from[j < dist ? j : j % dist];
      o += len;
    }
  }
  if (st == DAN_INFLATE_OK) {
    b.buf >>= b.cnt & 7; b.cnt &= ~7;                 // zlib trailer: Adler-32, big-endian, at the next byte boundary
    uint32_t a0, a1, a2, a3;
    if (!b.take(8, &a0) || !b.take(8, &a1) || !b.take(8, &a2) || !b.take(8, &a3)) st = DAN_INFLATE_E_INPUT;
    else if (o != slot_bytes) st = DAN_INFLATE_E_OUTPUT_SHORT;
    else {
      __syncwarp();
      // Adler-32 over 32 chunks, one per lane
      const uint64_t chunk = (slot_bytes + 31) / 32, s = min((uint64_t)lane * chunk, slot_bytes), m = min(chunk, slot_bytes - s);
      AdlerPart ad = adler_chunk(out, slot_bytes, s, m);
      for (int d = 16; d; d >>= 1) { ad.a += __shfl_xor_sync(0xffffffffu, ad.a, d); ad.b += __shfl_xor_sync(0xffffffffu, ad.b, d); }
      if (adler_value(ad.a, ad.b, slot_bytes) != ((a0 << 24) | (a1 << 16) | (a2 << 8) | a3)) st = DAN_INFLATE_E_ADLER;
    }
  }
  __syncwarp();
  if (st != DAN_INFLATE_OK) {                         // a failed stream leaves an all-zero slot
    for (uint64_t k = lane; k < slot_bytes; k += 32) out[k] = 0;
  }
  if (lane == 0) status[i] = st;
}

}  // namespace

int dan_inflate_launch(const uint8_t* src, const uint64_t* offsets, const uint32_t* lengths, int n, uint8_t* dst, uint64_t slot_bytes,
                       int32_t* status, cudaStream_t stream) {
  if (n == 0) return DAN_OK;
  inflate_kernel<<<(n + kWarps - 1) / kWarps, kWarps * 32, 0, stream>>>(src, offsets, lengths, n, dst, slot_bytes, status);
  DAN_CUDA_TRY(cudaGetLastError());
  return DAN_OK;
}

extern "C" int dan_inflate_device(const void* src, const uint64_t* offsets, const uint32_t* lengths, int n, void* dst, uint64_t slot_bytes,
                                  int32_t* status, void* stream) {
  if (n < 0) { dan_set_error("negative stream count"); return DAN_E_INVALID; }
  if (n == 0) return DAN_OK;
  if (!src || !offsets || !lengths || (!dst && slot_bytes) || !status) { dan_set_error("null pointer"); return DAN_E_INVALID; }
  return dan_inflate_launch(static_cast<const uint8_t*>(src), offsets, lengths, n, static_cast<uint8_t*>(dst), slot_bytes, status,
                            static_cast<cudaStream_t>(stream));
}
