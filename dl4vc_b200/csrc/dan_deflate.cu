// dan_deflate.cu — batched zlib (RFC 1950 / 1951) deflate on the GPU: n inputs of slot_bytes each into n complete zlib streams, the
// inverse of dan_inflate.cu; and the same deflate in BGZF framing (gzip members, RFC 1952, of <= 64 KB with the BC extra subfield):
// a buffer cut as bgzip cuts it, into 65280-byte pieces and a shorter last one, each piece one block with a CRC-32 and ISIZE.
//
// One CTA of 1024 threads per input. The input sits whole in shared memory beside a 2^14-entry hash table of 4-byte prefixes. The
// CTA walks the input in steps of 1024 positions, one position per thread:
//   1. match finding: each thread takes the longest match at its position among distance 1, the row strides 201 / 402 / 603 of the
//      record's [200][201] planes and the hash table's entry, which holds the latest position of an EARLIER step with the same
//      prefix hash; candidates are tried in increasing distance and only a strictly longer match replaces the best, so a tie keeps
//      the smaller distance. Then every position of the step enters the table with atomicMax, so each bucket holds the latest
//      position whatever the order of the atomics.
//   2. greedy parse: warp 0 walks the step's token starts 32 positions a round, a ballot finding the next match (one round per
//      match, one per 32 literals); a match that runs past the step carries its end into the next step.
//   3. coding: tokens starting in the same 16 KB of input form one dynamic-Huffman block.
// This runs twice. The first pass counts each block's symbols and builds its length-limited codes (15 bits, 7 for the code-length
// code; Moffat-Katajainen Huffman lengths in warp 0 over the symbols sorted by count, then miniz's Kraft repair), which gives the
// stream's exact size before any byte of it is written. If that exceeds the stored-block encoding, the stream is written as stored
// blocks; otherwise the second pass repeats the same matches and parse and writes the bits: a block-wide exclusive scan of the
// tokens' bit counts places each token, every thread ORs its bits into a shared-memory window, and the window's whole bytes go to
// the output slot after every step. Nothing depends on float arithmetic, atomic order or the batch, so a stream's bytes depend only
// on its input. The two containers differ only around the deflate blocks: the header, and an Adler-32 (chunk parts summed) or a CRC-32
// (chunk CRCs combined pairwise in a fixed tree), computed by the same one-chunk-per-thread split.
#include <cstdint>
#include <cuda_runtime.h>
#include "dan_internal.h"
#include "dan_zlib.cuh"

namespace {

constexpr int kThreads = 1024;
constexpr uint32_t kStep = kThreads;                 // positions per step, one per thread
constexpr uint32_t kMaxSlot = DAN_DEFLATE_MAX_SLOT;  // largest input: the shared-memory budget
constexpr int kHashBits = 14;
constexpr uint32_t kBlock = 16 * 1024;               // input positions whose tokens form one Huffman block
constexpr int kMaxBlocks = kMaxSlot / kBlock;
constexpr int kLitCodes = 286, kDistCodes = 30, kSyms = kLitCodes + kDistCodes;
constexpr int kWinWords = 2048;                      // bit window: one block header plus 1024 tokens of <= 48 bits fit
constexpr uint32_t kWindow = 32768, kMaxMatch = 258;
constexpr uint32_t kTok = 1u << 31;                  // mt[]: token start; bits 16..24 match length (0: literal), 0..15 distance

struct Smem {
  uint8_t in[kMaxSlot + 16];                         // the input; 16 zero bytes behind it for the word-wise compare
  int32_t hash[1 << kHashBits];                      // latest earlier position of each 4-byte prefix hash, -1 none
  uint32_t mt[kStep];                                // the step's matches, then its token starts
  uint32_t win[kWinWords];
  uint32_t hist[kSyms];                              // symbol counts of the current block: literal/length, then distance
  uint8_t lens[kMaxBlocks][kSyms];                   // code lengths of each block (first pass), read by the second
  uint16_t code[kSyms];                              // bit-reversed canonical codes of the current block
  uint8_t len_sym[kMaxMatch + 1];                    // match length -> length symbol - 257
  uint8_t dist_sym[512];                             // distance - 1 -> distance symbol, zlib's two-level table
  // Huffman construction scratch (warp 0)
  uint32_t fr[kLitCodes], key[kLitCodes], num[33];
  uint16_t sym[kLitCodes];
  // block header: run-length coded code lengths (symbol | extra << 5) and the code-length code
  uint16_t rle[kSyms];
  uint32_t clf[19];
  uint8_t cl_len[19];
  uint16_t cl_code[19];
  uint32_t warp_sum[32];
  uint64_t adler_a[32], adler_b[32];
  uint32_t crc_part[32], crc_len[32];                // CRC-32 of each warp's chunks and their length
  uint64_t total_bits;
  uint32_t carry, wbit, outpos, nrle, nlit, ndist;
};

static_assert(sizeof(Smem) <= 227 * 1024, "the deflate CTA's shared memory exceeds the 227 KB an sm_100a block may use");

__device__ __forceinline__ uint32_t load4(const uint8_t* in, uint32_t p) {      // bytes p..p+3, little-endian, from aligned words
  const uint32_t* w = reinterpret_cast<const uint32_t*>(in) + (p >> 2);
  return __funnelshift_r(w[0], w[1], (p & 3) * 8);
}

__device__ __forceinline__ uint32_t hash4(const uint8_t* in, uint32_t p) { return (load4(in, p) * 2654435761u) >> (32 - kHashBits); }

// length of the common prefix of in[a..] and in[b..], at most maxlen
__device__ __forceinline__ uint32_t match_len(const uint8_t* in, uint32_t a, uint32_t b, uint32_t maxlen) {
  for (uint32_t k = 0; k < maxlen; k += 4) {
    const uint32_t x = load4(in, a + k) ^ load4(in, b + k);
    if (x) return min(maxlen, k + ((__ffs(x) - 1) >> 3));
  }
  return maxlen;
}

__device__ __forceinline__ uint32_t dist_symbol(const Smem& sm, uint32_t d) {
  return d <= 256 ? sm.dist_sym[d - 1] : sm.dist_sym[256 + ((d - 1) >> 7)];
}

// the best match at p (packed as in mt[], 0 for none); positions before the current step are in the hash table
__device__ uint32_t find_match(const Smem& sm, uint32_t p, uint32_t n) {
  const uint32_t maxlen = min(kMaxMatch, n - p);
  if (maxlen < 3) return 0;
  uint32_t hd = 0;
  if (n - p >= 4) {
    const int q = sm.hash[hash4(sm.in, p)];
    if (q >= 0 && p - (uint32_t)q <= kWindow) hd = p - (uint32_t)q;
  }
  uint32_t best = 0, best_d = 0;
  auto tryd = [&](uint32_t d) {
    if (best < maxlen && sm.in[p + best] == sm.in[p - d + best]) {
      const uint32_t l = match_len(sm.in, p - d, p, maxlen);
      if (l > best) { best = l; best_d = d; }
    }
  };
  constexpr uint32_t kRows[4] = {1, 201, 402, 603};
  uint32_t prev = 0;
#pragma unroll
  for (int c = 0; c < 5; ++c) {
    const uint32_t sd = c < 4 ? kRows[c] : 0xffffffffu;
    if (hd > prev && hd < sd) tryd(hd);
    if (c < 4 && sd <= p) tryd(sd);
    prev = sd;
  }
  return best >= 3 ? (best << 16) | best_d : 0;
}

// warp 0: mark the token starts of [lo, hi) in mt[], starting at sm.carry, and carry the next token start on
__device__ void walk(Smem& sm, uint32_t lo, uint32_t hi, int lane) {
  uint32_t cur = sm.carry;
  while (cur < hi) {
    const uint32_t p = cur + lane;
    const uint32_t m = p < hi ? sm.mt[p - lo] : 0;
    const uint32_t has = __ballot_sync(0xffffffffu, m != 0);
    const int f = has ? __ffs(has) - 1 : 32;          // lanes before f are literals, lane f the next match
    if (p < hi && lane <= f) sm.mt[p - lo] = m | kTok;
    const uint32_t len = __shfl_sync(0xffffffffu, m, f & 31) >> 16;
    cur = f < 32 ? cur + f + len : min(cur + 32, hi);
  }
  if (lane == 0) sm.carry = cur;
  __syncwarp();
}

__device__ __forceinline__ void put_bits(uint32_t* win, uint32_t pos, uint32_t v, int nbits) {   // nbits <= 32, v < 2^nbits
  if (!nbits) return;
  const uint32_t w = pos >> 5, sh = pos & 31;
  atomicOr(&win[w], v << sh);
  if (sh + nbits > 32) atomicOr(&win[w + 1], v >> (32 - sh));
}

// In-place Moffat-Katajainen: A[0, n) ascending counts -> Huffman code lengths of the same symbols (n >= 2).
__device__ void huffman_lengths(uint32_t* A, int n) {
  A[0] += A[1];
  int root = 0, leaf = 2;
  for (int next = 1; next < n - 1; ++next) {
    if (leaf >= n || A[root] < A[leaf]) { A[next] = A[root]; A[root++] = next; } else A[next] = A[leaf++];
    if (leaf >= n || (root < next && A[root] < A[leaf])) { A[next] += A[root]; A[root++] = next; } else A[next] += A[leaf++];
  }
  A[n - 2] = 0;
  for (int next = n - 3; next >= 0; --next) A[next] = A[A[next]] + 1;
  int avail = 1, used = 0, depth = 0, next = n - 1;
  root = n - 2;
  while (avail > 0) {
    while (root >= 0 && (int)A[root] == depth) { ++used; --root; }
    while (avail > used) { A[next--] = depth; --avail; }
    avail = 2 * used; ++depth; used = 0;
  }
}

// warp 0: code lengths <= maxbits of freq[0, n) into lens[0, n), 0 for an unused symbol. When fewer than two symbols are used, unused
// ones get a count of 1 until two are, so that every code is complete (the code-length code must be; for the others it costs nothing).
__device__ void build_lengths(Smem& sm, const uint32_t* freq, int n, int maxbits, uint8_t* lens, int lane) {
  for (int s = lane; s < n; s += 32) { sm.fr[s] = freq[s]; lens[s] = 0; }
  __syncwarp();
  int used = 0;
  if (lane == 0) {
    for (int s = 0; s < n; ++s) used += sm.fr[s] != 0;
    for (int s = 0; used < 2 && s < n; ++s) if (!sm.fr[s]) { sm.fr[s] = 1; ++used; }
  }
  used = __shfl_sync(0xffffffffu, used, 0);
  __syncwarp();
  for (int s = lane; s < n; s += 32) {                 // rank by (count, symbol): a fixed order whatever the lanes do
    const uint32_t f = sm.fr[s];
    if (!f) continue;
    int r = 0;
    for (int t = 0; t < n; ++t) { const uint32_t g = sm.fr[t]; r += g && (g < f || (g == f && t < s)); }
    sm.sym[r] = (uint16_t)s; sm.key[r] = f;
  }
  __syncwarp();
  if (lane == 0) {
    huffman_lengths(sm.key, used);
    for (int l = 0; l <= 32; ++l) sm.num[l] = 0;
    for (int k = 0; k < used; ++k) sm.num[min(sm.key[k], 32u)]++;
    for (int l = maxbits + 1; l <= 32; ++l) sm.num[maxbits] += sm.num[l];
    uint32_t total = 0;
    for (int l = maxbits; l > 0; --l) total += sm.num[l] << (maxbits - l);
    while (total != (1u << maxbits)) {                 // over-subscribed after the clamp: lengthen codes until the Kraft sum is 1
      sm.num[maxbits]--;
      for (int l = maxbits - 1; l > 0; --l)
        if (sm.num[l]) { sm.num[l]--; sm.num[l + 1] += 2; break; }
      --total;
    }
    int j = 0;                                         // the most frequent symbols take the shortest codes
    for (int l = 1; l <= maxbits; ++l)
      for (uint32_t k = sm.num[l]; k > 0; --k) lens[sm.sym[used - 1 - j++]] = (uint8_t)l;
  }
  __syncwarp();
}

// one thread: bit-reversed canonical codes of lens[0, n) (RFC 1951 §3.2.2)
__device__ void canonical_codes(Smem& sm, const uint8_t* lens, int n, uint16_t* code) {
  uint32_t *cnt = sm.num, *next = sm.num + 16;
  for (int l = 0; l < 16; ++l) cnt[l] = 0;
  for (int s = 0; s < n; ++s) cnt[lens[s]]++;
  cnt[0] = 0;
  uint32_t c = 0;
  for (int l = 1; l < 16; ++l) { c = (c + cnt[l - 1]) << 1; next[l] = c; }
  for (int s = 0; s < n; ++s) {
    const int l = lens[s];
    if (l) code[s] = (uint16_t)(__brev(next[l]++) >> (32 - l));
  }
}

// warp 0: the dynamic block header of the code lengths `lens`. Returns its bit count (on lane 0); with kEmit also writes it at sm.wbit.
template <bool kEmit>
__device__ uint64_t block_header(Smem& sm, const uint8_t* lens, bool final_block, int lane) {
  if (lane == 0) {
    int nlit = kLitCodes, ndist = kDistCodes;
    while (nlit > 257 && !lens[nlit - 1]) --nlit;
    while (ndist > 1 && !lens[kLitCodes + ndist - 1]) --ndist;
    for (int k = 0; k < 19; ++k) sm.clf[k] = 0;
    auto at = [&](int k) { return k < nlit ? lens[k] : lens[kLitCodes + k - nlit]; };
    int nr = 0;
    auto emit = [&](int s, int extra) { sm.rle[nr++] = (uint16_t)(s | extra << 5); sm.clf[s]++; };
    const int total = nlit + ndist;
    for (int k = 0; k < total;) {                      // runs of one length: 16 repeats the previous length, 17 / 18 code zeros
      const int v = at(k);
      int run = 1;
      while (k + run < total && at(k + run) == v) ++run;
      int r = run;
      if (v == 0) {
        while (r >= 11) { const int c = min(r, 138); emit(18, c - 11); r -= c; }
        if (r >= 3) { emit(17, r - 3); r = 0; }
      } else {
        emit(v, 0); --r;
        while (r >= 3) { const int c = min(r, 6); emit(16, c - 3); r -= c; }
      }
      for (; r > 0; --r) emit(v, 0);
      k += run;
    }
    sm.nrle = nr; sm.nlit = nlit; sm.ndist = ndist;
  }
  __syncwarp();
  build_lengths(sm, sm.clf, 19, 7, sm.cl_len, lane);
  uint64_t bits = 0;
  if (lane == 0) {
    int hclen = 19;
    while (hclen > 4 && !sm.cl_len[kClOrder[hclen - 1]]) --hclen;
    auto ebits = [](int s) { return s == 16 ? 2 : s == 17 ? 3 : 7; };
    bits = 3 + 5 + 5 + 4 + 3 * hclen;
    for (uint32_t r = 0; r < sm.nrle; ++r) {
      const int s = sm.rle[r] & 31;
      bits += sm.cl_len[s] + (s >= 16 ? ebits(s) : 0);
    }
    if (kEmit) {
      canonical_codes(sm, sm.cl_len, 19, sm.cl_code);
      uint32_t pos = sm.wbit;
      put_bits(sm.win, pos, (final_block ? 1u : 0u) | 2u << 1, 3); pos += 3;
      put_bits(sm.win, pos, sm.nlit - 257, 5); pos += 5;
      put_bits(sm.win, pos, sm.ndist - 1, 5); pos += 5;
      put_bits(sm.win, pos, hclen - 4, 4); pos += 4;
      for (int k = 0; k < hclen; ++k) { put_bits(sm.win, pos, sm.cl_len[kClOrder[k]], 3); pos += 3; }
      for (uint32_t r = 0; r < sm.nrle; ++r) {
        const int s = sm.rle[r] & 31, e = sm.rle[r] >> 5;
        put_bits(sm.win, pos, sm.cl_code[s], sm.cl_len[s]); pos += sm.cl_len[s];
        if (s >= 16) { put_bits(sm.win, pos, e, ebits(s)); pos += ebits(s); }
      }
      sm.wbit = pos;
    }
  }
  __syncwarp();
  return bits;
}

// block-wide exclusive scan of v; *total receives the sum
__device__ uint32_t block_scan(Smem& sm, uint32_t v, uint32_t* total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t incl = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) { const uint32_t x = __shfl_up_sync(0xffffffffu, incl, d); if (lane >= d) incl += x; }
  if (lane == 31) sm.warp_sum[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    uint32_t w = sm.warp_sum[lane];
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const uint32_t x = __shfl_up_sync(0xffffffffu, w, d); if (lane >= d) w += x; }
    sm.warp_sum[lane] = w;
  }
  __syncthreads();
  *total = sm.warp_sum[31];
  const uint32_t base = warp ? sm.warp_sum[warp - 1] : 0;
  __syncthreads();                                     // warp_sum is free again on return
  return base + incl - v;
}

// the window's whole bytes to out[outpos..] (never at or past `cap`); its last partial byte moves to the front
__device__ void flush(Smem& sm, uint8_t* out, uint32_t cap) {
  __syncthreads();
  const uint32_t wb = sm.wbit, nbytes = wb >> 3, pos = sm.outpos;
  const uint8_t* w8 = reinterpret_cast<const uint8_t*>(sm.win);
  for (uint32_t k = threadIdx.x; k < nbytes; k += kThreads)
    if (pos + k < cap) out[pos + k] = w8[k];
  const uint32_t tail = w8[nbytes];
  __syncthreads();
  for (uint32_t k = threadIdx.x; k <= (wb >> 5); k += kThreads) sm.win[k] = 0;
  __syncthreads();
  if (threadIdx.x == 0) { sm.win[0] = tail; sm.outpos = pos + nbytes; sm.wbit = wb & 7; }
  __syncthreads();
}

// One pass over the input (see the file comment). kEmit = false: each block's code lengths into sm.lens and the stream's deflate bit
// count into sm.total_bits. kEmit = true: the bits behind the 2-byte zlib header, whole bytes in out[2, sm.outpos), sm.wbit bits left
// in sm.win[0].
template <bool kEmit>
__device__ void deflate_pass(Smem& sm, uint32_t n, uint8_t* out, uint32_t cap) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int k = tid; k < (1 << kHashBits); k += kThreads) sm.hash[k] = -1;
  if (kEmit) for (int k = tid; k < kWinWords; k += kThreads) sm.win[k] = 0;
  if (tid == 0) { sm.carry = 0; sm.wbit = 0; sm.outpos = 2; sm.total_bits = 0; }
  const int nblocks = n ? (int)((n + kBlock - 1) / kBlock) : 1;
  __syncthreads();
  for (int b = 0; b < nblocks; ++b) {
    const uint32_t blo = b * kBlock, bhi = min(n, blo + kBlock);
    uint8_t* lens = sm.lens[b];
    if (!kEmit) {
      for (int k = tid; k < kSyms; k += kThreads) sm.hist[k] = k == 256;       // the end-of-block code
    } else if (warp == 0) {
      if (lane == 0) { canonical_codes(sm, lens, kLitCodes, sm.code); canonical_codes(sm, lens + kLitCodes, kDistCodes, sm.code + kLitCodes); }
      __syncwarp();
      block_header<true>(sm, lens, b == nblocks - 1, lane);
    }
    __syncthreads();
    for (uint32_t lo = blo; lo < bhi; lo += kStep) {
      const uint32_t hi = min(bhi, lo + kStep), p = lo + tid;
      sm.mt[tid] = p < hi ? find_match(sm, p, n) : 0;
      __syncthreads();
      if (p < hi && p + 4 <= n) atomicMax(&sm.hash[hash4(sm.in, p)], (int)p);
      if (warp == 0) walk(sm, lo, hi, lane);
      __syncthreads();
      const uint32_t t = sm.mt[tid], len = (t >> 16) & 511, d = t & 0xffff;
      const bool tok = (t & kTok) != 0;
      if (!kEmit) {
        if (tok) {
          if (!len) {
            atomicAdd(&sm.hist[sm.in[p]], 1u);
          } else {
            atomicAdd(&sm.hist[257 + sm.len_sym[len]], 1u);
            atomicAdd(&sm.hist[kLitCodes + dist_symbol(sm, d)], 1u);
          }
        }
      } else {
        uint32_t nbits = 0, ls = 0, ds = 0;
        if (tok) {
          if (!len) {
            nbits = lens[sm.in[p]];
          } else {
            ls = sm.len_sym[len]; ds = dist_symbol(sm, d);
            nbits = lens[257 + ls] + kLenExtra[ls] + lens[kLitCodes + ds] + kDistExtra[ds];
          }
        }
        const uint32_t base = sm.wbit;
        uint32_t total;
        const uint32_t at = base + block_scan(sm, nbits, &total);
        if (tok) {
          if (!len) {
            put_bits(sm.win, at, sm.code[sm.in[p]], lens[sm.in[p]]);
          } else {
            const int l1 = lens[257 + ls], e1 = kLenExtra[ls], l2 = lens[kLitCodes + ds];
            put_bits(sm.win, at, sm.code[257 + ls] | (len - kLenBase[ls]) << l1, l1 + e1);
            put_bits(sm.win, at + l1 + e1, sm.code[kLitCodes + ds] | (d - kDistBase[ds]) << l2, l2 + kDistExtra[ds]);
          }
        }
        if (tid == 0) sm.wbit = base + total;
        flush(sm, out, cap);
      }
    }
    __syncthreads();
    if (!kEmit) {
      if (warp == 0) {
        build_lengths(sm, sm.hist, kLitCodes, 15, lens, lane);
        build_lengths(sm, sm.hist + kLitCodes, kDistCodes, 15, lens + kLitCodes, lane);
        uint64_t bits = 0;
        for (int s = lane; s < kSyms; s += 32) {
          const int extra = s >= kLitCodes ? kDistExtra[s - kLitCodes] : s > 256 ? kLenExtra[s - 257] : 0;
          bits += (uint64_t)sm.hist[s] * (lens[s] + extra);
        }
        for (int o = 16; o; o >>= 1) bits += __shfl_xor_sync(0xffffffffu, bits, o);
        bits += block_header<false>(sm, lens, b == nblocks - 1, lane);
        if (lane == 0) sm.total_bits += bits;
      }
    } else {
      if (tid == 0) { put_bits(sm.win, sm.wbit, sm.code[256], lens[256]); sm.wbit += lens[256]; }
      flush(sm, out, cap);
    }
    __syncthreads();
  }
}

// The container around the deflate blocks: a zlib stream (2-byte header, big-endian Adler-32) or a BGZF block (18-byte gzip header with
// the BC subfield, little-endian CRC-32 and ISIZE).
enum class Container { kZlib, kBgzf };

// CTA i compresses src[i * in_stride, min((i + 1) * in_stride, in_total)) into dst + i * out_stride. The stream is written as stored
// blocks when the deflate blocks would be longer, so out_stride >= the stored size of in_stride bytes keeps every write in the slot.
template <Container kC>
__global__ void __launch_bounds__(kThreads, 1) deflate_kernel(const uint8_t* __restrict__ src, uint64_t in_stride, uint64_t in_total,
                                                             uint8_t* __restrict__ dst, uint64_t out_stride, uint32_t* __restrict__ lengths,
                                                             int32_t* __restrict__ status) {
  constexpr uint32_t kHead = kC == Container::kZlib ? 2 : 18, kTail = kC == Container::kZlib ? 4 : 8;
  extern __shared__ __align__(16) uint8_t smem_raw[];
  Smem& sm = *reinterpret_cast<Smem*>(smem_raw);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint64_t i = blockIdx.x;
  if (in_stride > kMaxSlot) {                        // the launchers refuse these; kept so that no write can leave shared memory
    if (tid == 0) { lengths[i] = 0; status[i] = DAN_DEFLATE_E_UNSUPPORTED; }
    return;
  }
  const uint32_t n = (uint32_t)min(in_stride, in_total - i * in_stride);
  const uint8_t* in_g = src + i * in_stride;
  uint8_t* out = dst + i * out_stride;
  uint8_t* body = out + (kHead - 2);                 // deflate_pass and the stored blocks write from body[2] on, behind the header
  for (uint32_t k = tid; k < n + 16; k += kThreads) sm.in[k] = k < n ? in_g[k] : 0;
  for (int e = tid; e < 512 + (int)kMaxMatch + 1; e += kThreads) {
    if (e < 512) {                                   // zlib's d_code: entry d - 1 for d <= 256, 256 + ((d - 1) >> 7) above
      const uint32_t d = e < 256 ? e + 1 : ((uint32_t)(e - 256) << 7) + 1;
      int s = 29;
      while (s > 0 && kDistBase[s] > d) --s;
      sm.dist_sym[e] = (uint8_t)s;
    } else {
      const uint32_t l = e - 512;
      int s = 28;
      while (s > 0 && kLenBase[s] > l) --s;
      sm.len_sym[l] = (uint8_t)s;
    }
  }
  __syncthreads();
  // the checksum: one chunk per thread; Adler-32 parts add up, CRC-32 parts combine pairwise in a fixed tree
  {
    const uint32_t chunk = (n + kThreads - 1) / kThreads, s = min(tid * chunk, n), m = min(chunk, n - s);
    if (kC == Container::kZlib) {
      AdlerPart ad = adler_chunk(sm.in, n, s, m);
      for (int d = 16; d; d >>= 1) { ad.a += __shfl_xor_sync(0xffffffffu, ad.a, d); ad.b += __shfl_xor_sync(0xffffffffu, ad.b, d); }
      if (lane == 0) { sm.adler_a[warp] = ad.a; sm.adler_b[warp] = ad.b; }
    } else {
      uint32_t crc = crc32_chunk(sm.in, s, m), len = m;
      for (int d = 1; d < 32; d <<= 1) {             // lane l (a multiple of 2d) takes on lanes [l + d, l + 2d)
        const uint32_t c2 = __shfl_down_sync(0xffffffffu, crc, d), l2 = __shfl_down_sync(0xffffffffu, len, d);
        if (!(lane & (2 * d - 1))) { crc = crc32_combine(crc, c2, l2); len += l2; }
      }
      if (lane == 0) { sm.crc_part[warp] = crc; sm.crc_len[warp] = len; }
    }
  }
  deflate_pass<false>(sm, n, body, 0);
  uint32_t check = 0;
  if (kC == Container::kZlib) {
    if (tid == 0) {
      uint64_t a = 0, b = 0;
      for (int w = 0; w < 32; ++w) { a += sm.adler_a[w]; b += sm.adler_b[w]; }
      check = adler_value(a, b, n);
    }
  } else if (warp == 0) {                            // the same tree over the 32 warps' parts
    uint32_t crc = sm.crc_part[lane], len = sm.crc_len[lane];
    for (int d = 1; d < 32; d <<= 1) {
      const uint32_t c2 = __shfl_down_sync(0xffffffffu, crc, d), l2 = __shfl_down_sync(0xffffffffu, len, d);
      if (!(lane & (2 * d - 1))) { crc = crc32_combine(crc, c2, l2); len += l2; }
    }
    check = crc;
  }
  const uint32_t nb = n ? (n + 65534) / 65535 : 1;   // stored blocks of the input
  const uint64_t stored = kHead + 5ull * nb + n + kTail;
  const uint64_t zbytes = kHead + (sm.total_bits + 7) / 8 + kTail;
  uint64_t len;                                      // bytes of body: 2 + the deflate blocks
  if (zbytes <= stored) {
    deflate_pass<true>(sm, n, body, (uint32_t)(stored - kTail - (kHead - 2)));
    len = sm.outpos;
    if (tid == 0 && sm.wbit) body[len] = (uint8_t)sm.win[0];
    len += sm.wbit ? 1 : 0;
  } else {                                           // stored blocks of <= 65535 bytes: BFINAL/BTYPE byte, LEN, NLEN, the bytes
    for (uint32_t k = tid; k < n; k += kThreads) body[2 + 5 * (k / 65535 + 1) + k] = sm.in[k];
    if ((uint32_t)tid < nb) {
      const uint32_t ln = min(65535u, n - tid * 65535u), o = 2 + tid * (65535u + 5);
      body[o] = tid == (int)nb - 1;
      body[o + 1] = ln & 255; body[o + 2] = ln >> 8; body[o + 3] = ~ln & 255; body[o + 4] = (~ln >> 8) & 255;
    }
    len = 2 + 5ull * nb + n;
  }
  if (tid == 0) {
    uint8_t* t = body + len;
    if (kC == Container::kZlib) {                    // zlib header (deflate, 32 KB window, FCHECK) and the big-endian Adler-32
      out[0] = 0x78; out[1] = 0x01;
      t[0] = check >> 24; t[1] = (check >> 16) & 255; t[2] = (check >> 8) & 255; t[3] = check & 255;
    } else {                                         // gzip header: deflate, FEXTRA, MTIME 0, XFL 0, OS 255, XLEN 6, BC, BSIZE
      const uint32_t bsize = (uint32_t)(kHead - 2 + len + kTail - 1);
      const uint8_t h[16] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 'B', 'C', 2, 0};
      for (int k = 0; k < 16; ++k) out[k] = h[k];
      out[16] = bsize & 255; out[17] = bsize >> 8;
      for (int k = 0; k < 4; ++k) { t[k] = (check >> (8 * k)) & 255; t[4 + k] = (n >> (8 * k)) & 255; }
    }
    lengths[i] = (uint32_t)(kHead - 2 + len + kTail);
    status[i] = DAN_DEFLATE_OK;
  }
}

// offsets[i] = lengths[0] + ... + lengths[i - 1] for i <= n, one CTA
__global__ void __launch_bounds__(1024) compact_offsets_kernel(const uint32_t* __restrict__ lengths, int n, uint64_t* __restrict__ offsets) {
  __shared__ uint64_t wsum[32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  uint64_t carry = 0;
  for (int lo = 0; lo < n; lo += 1024) {
    const uint64_t v = lo + tid < n ? lengths[lo + tid] : 0;
    uint64_t incl = v;
    for (int d = 1; d < 32; d <<= 1) { const uint64_t x = __shfl_up_sync(0xffffffffu, incl, d); if (lane >= d) incl += x; }
    if (lane == 31) wsum[warp] = incl;
    __syncthreads();
    uint64_t before = 0, tile = 0;
    for (int w = 0; w < 32; ++w) { before += w < warp ? wsum[w] : 0; tile += wsum[w]; }
    if (lo + tid < n) offsets[lo + tid] = carry + before + incl - v;
    carry += tile;
    __syncthreads();
  }
  if (tid == 0) offsets[n] = carry;
}

__global__ void compact_copy_kernel(const uint8_t* __restrict__ slots, uint64_t stride, const uint32_t* __restrict__ lengths,
                                    const uint64_t* __restrict__ offsets, uint8_t* __restrict__ dst) {
  const uint64_t i = blockIdx.x;
  const uint8_t* s = slots + i * stride;
  uint8_t* d = dst + offsets[i];
  const uint64_t len = min((uint64_t)lengths[i], stride);
  for (uint64_t k = threadIdx.x; k < len; k += blockDim.x) d[k] = s[k];
}

// dan_deflate_compact and dan_bgzf_compact: the outputs of n slots `stride` bytes apart, back to back
int compact(const void* slots, uint64_t stride, const uint32_t* lengths, int n, void* dst, uint64_t* offsets, void* stream) {
  if (n < 0) { dan_set_error("negative stream count"); return DAN_E_INVALID; }
  if (!offsets) { dan_set_error("null pointer"); return DAN_E_INVALID; }
  if (n > 0 && (!slots || !lengths || !dst)) { dan_set_error("null pointer"); return DAN_E_INVALID; }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  compact_offsets_kernel<<<1, 1024, 0, st>>>(lengths, n, offsets);
  DAN_CUDA_TRY(cudaGetLastError());
  if (n == 0) return DAN_OK;
  compact_copy_kernel<<<n, 256, 0, st>>>(static_cast<const uint8_t*>(slots), stride, lengths, offsets, static_cast<uint8_t*>(dst));
  DAN_CUDA_TRY(cudaGetLastError());
  return DAN_OK;
}

DanSmemAttr g_deflate_smem, g_bgzf_smem;

}  // namespace

extern "C" size_t dan_deflate_bound(uint64_t slot_bytes) {
  const uint64_t blocks = slot_bytes ? (slot_bytes + 65534) / 65535 : 1;
  return (size_t)(slot_bytes + 5 * blocks + 6);
}

extern "C" int dan_deflate_device(const void* src, int n, uint64_t slot_bytes, void* dst, uint32_t* lengths, int32_t* status, void* stream) {
  if (n < 0) { dan_set_error("negative input count"); return DAN_E_INVALID; }
  if (slot_bytes > kMaxSlot) {
    dan_set_error("slot_bytes %llu exceeds the deflate kernel's %u (the input must fit in shared memory)", (unsigned long long)slot_bytes, kMaxSlot);
    return DAN_E_UNSUPPORTED;
  }
  if (n == 0) return DAN_OK;
  if ((!src && slot_bytes) || !dst || !lengths || !status) { dan_set_error("null pointer"); return DAN_E_INVALID; }
  DAN_CUDA_TRY(g_deflate_smem.ensure(deflate_kernel<Container::kZlib>, sizeof(Smem)));
  deflate_kernel<Container::kZlib><<<n, kThreads, sizeof(Smem), static_cast<cudaStream_t>(stream)>>>(
      static_cast<const uint8_t*>(src), slot_bytes, (uint64_t)n * slot_bytes, static_cast<uint8_t*>(dst), dan_deflate_bound(slot_bytes),
      lengths, status);
  DAN_CUDA_TRY(cudaGetLastError());
  return DAN_OK;
}

extern "C" int dan_deflate_compact(const void* slots, const uint32_t* lengths, int n, uint64_t slot_bytes, void* dst, uint64_t* offsets,
                                   void* stream) {
  return compact(slots, dan_deflate_bound(slot_bytes), lengths, n, dst, offsets, stream);
}

static_assert(DAN_BGZF_MAX_INPUT <= kMaxSlot && 18 + 5 + DAN_BGZF_MAX_INPUT + 8 <= DAN_BGZF_MAX_BLOCK,
              "a BGZF piece must fit in shared memory and its stored encoding in one slot");

extern "C" int dan_bgzf_compress_device(const void* src, uint64_t bytes, void* dst, uint32_t* block_lengths, int32_t* status, void* stream) {
  if (bytes == 0) return DAN_OK;
  if (!src || !dst || !block_lengths || !status) { dan_set_error("null pointer"); return DAN_E_INVALID; }
  const uint64_t n = (bytes + DAN_BGZF_MAX_INPUT - 1) / DAN_BGZF_MAX_INPUT;
  if (n > 0x7fffffffull) { dan_set_error("%llu bytes make more than 2^31 - 1 BGZF blocks", (unsigned long long)bytes); return DAN_E_INVALID; }
  DAN_CUDA_TRY(g_bgzf_smem.ensure(deflate_kernel<Container::kBgzf>, sizeof(Smem)));
  deflate_kernel<Container::kBgzf><<<(unsigned)n, kThreads, sizeof(Smem), static_cast<cudaStream_t>(stream)>>>(
      static_cast<const uint8_t*>(src), DAN_BGZF_MAX_INPUT, bytes, static_cast<uint8_t*>(dst), DAN_BGZF_MAX_BLOCK, block_lengths, status);
  DAN_CUDA_TRY(cudaGetLastError());
  return DAN_OK;
}

extern "C" int dan_bgzf_compact(const void* slots, const uint32_t* lengths, int n, void* dst, uint64_t* offsets, void* stream) {
  return compact(slots, DAN_BGZF_MAX_BLOCK, lengths, n, dst, offsets, stream);
}
