// dan_bf16.cu — tcgen05 implementation of the DAN forward (bf16 operands, fp32 accumulation in TMEM).
//
// Activations are stored "chunk-major": for each group of 8 channels (one 16-byte piece per row) the rows of the
// pass form a dense array:   X[kc][row][8]  (bf16), rows = (candidate, read, position) with `gap` zero rows between
// reads (RowGeom). A tile of 128 consecutive rows (+ halo) of one channel chunk is therefore ONE contiguous run in
// HBM, moved by a single bulk async copy, and lands in shared memory exactly in the row-linear UMMA operand layout
// described in tcgen05_ptx.cuh — the three dilated taps of a conv layer are three start addresses on that tile.
//
// Kernels
//   dan_stack_kernel   (dan_stack.cuh) the fused, persistent conv-stack kernel: encoder prologue, all conv layers of a segment in
//                      shared memory, read-axis max / sum by TMA bulk reductions — the PROD path.
//   dan_layer_kernel   (dan_layerwise.cuh) one conv layer per launch: fallback for shapes the fused kernel does not take.
//   tma_gemm_kernel    (dan_gemm.cuh) TMA-fed batched GEMM: highway compression (1x201) conv as one K=6432 GEMM over reads,
//                      pool bias map, post-pool Linear (pool_combine_dimension > 0), FC trunk, heads.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>
#include "dan_kernels_common.cuh"
#include "tcgen05_ptx.cuh"

namespace {

using namespace ptx;

constexpr int kC = 128;               // channels (bf16 path is specialised for the shipped width)
constexpr int kKC = kC / 8;           // 16-byte pieces per row
constexpr int kLead = 8;              // zero rows in front of every row matrix (>= largest dilation)
// Every CTA of the fused kernel streams the same few hundred KB of layer weights at about the same time; CTA c reads replica
// c % kWeightReplicas so that the reads spread over more L2 slices. (With per-slot rings 16 copies helped; with the shared ring,
// the evict-last L2 policy and two producer threads 1-4 copies measure the same and 16+ slightly worse.)
constexpr int kWeightReplicas = 4;

// =====================================================================================================
// Encoder (bf16, chunk-major output)
// =====================================================================================================
__global__ void __launch_bounds__(256) encode_rows_bf16_kernel(EncodeParams p, long cand0, uint4* __restrict__ out, long kstride) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const long cand = cand0 + blockIdx.x;
  EncodeSmem s = encode_stage(p, cand, smem_raw);
  const int rows = p.g.R * p.g.pitch;
  const int kcs = p.CinPad / 8;
  const long row0 = (long)blockIdx.x * rows;
  for (int idx = threadIdx.x; idx < rows * kcs; idx += blockDim.x) {
    const int kc = idx / rows, row = idx - kc * rows;
    const int r = row / p.g.pitch, pp = row - r * p.g.pitch;
    uint4 v = make_uint4(0, 0, 0, 0);
    if (pp < p.g.P) {
      float f[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) f[j] = (kc * 8 + j < p.Cin) ? encode_channel(p, s, kc * 8 + j, pp, r) : 0.f;
      v.x = pack_bf16x2(f[0], f[1]); v.y = pack_bf16x2(f[2], f[3]); v.z = pack_bf16x2(f[4], f[5]); v.w = pack_bf16x2(f[6], f[7]);
    }
    out[kc * kstride + kLead + row0 + row] = v;
  }
}


// bf16(E[tok] + pe[p]) for every (position, token): the read / reference embedding channels of the conv-1 input (model.py:450-451,
// 463-470,506-507) as three 16-byte pieces per entry (channels 0-7 | 8-15 | 16-19 + zero fill). Built once per weight load; the fused
// kernel's encoder prologue (dan_stack.cuh) assembles the input planes of a read from it.
__global__ void enc_table_kernel(const float* __restrict__ emb, const float* __restrict__ pe, int P, int D, uint4* __restrict__ tab) {
  const int total = P * DAN_VOCAB * 24;
  __nv_bfloat16* t = reinterpret_cast<__nv_bfloat16*>(tab);
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int c = i % 24, tok = (i / 24) % DAN_VOCAB, pp = i / (24 * DAN_VOCAB);
    t[i] = __float2bfloat16_rn(c < D ? emb[tok * D + c] + pe[pp * D + c] : 0.f);
  }
}

}  // namespace
#include "dan_layerwise.cuh"
#include "dan_stack.cuh"
#include "dan_gemm.cuh"
namespace {

// =====================================================================================================
// Elementwise / reduction helpers on chunk-major bf16
// =====================================================================================================
__device__ __forceinline__ void unpack8(const uint4& v, float (&f)[8]) {
  f[0] = bf16_lo(v.x); f[1] = bf16_hi(v.x); f[2] = bf16_lo(v.y); f[3] = bf16_hi(v.y);
  f[4] = bf16_lo(v.z); f[5] = bf16_hi(v.z); f[6] = bf16_lo(v.w); f[7] = bf16_hi(v.w);
}
__device__ __forceinline__ uint4 pack8(const float (&f)[8]) {
  return make_uint4(pack_bf16x2(f[0], f[1]), pack_bf16x2(f[2], f[3]), pack_bf16x2(f[4], f[5]), pack_bf16x2(f[6], f[7]));
}

// loads in flight per thread of the pooling kernels: they run as one 64-thread CTA per SM beside the persistent stack kernel
// (4096 spare registers per SM), so memory-level parallelism has to come from the thread itself
constexpr int kPoolUnroll = 8;
constexpr size_t kBmapBytesPerCand = (size_t)kStkBmapPerCand * 16;

// ---- layer-wise fallback path: pool[cand][c/8][p][c%8] = mean over reads (fp32)   (model.py:772) ----
__global__ void __launch_bounds__(64) pool_mean_bf16_kernel(const uint4* __restrict__ h, long kstride, float* __restrict__ pool, RowGeom g) {
  const int cand = blockIdx.y, kc = blockIdx.z;
  const int pp = blockIdx.x * blockDim.x + threadIdx.x;
  if (pp >= g.P) return;
  float s[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  const uint4* src = h + kc * kstride + kLead + (long)cand * g.R * g.pitch + pp;
  int r = 0;
  for (; r + kPoolUnroll <= g.R; r += kPoolUnroll) {
    uint4 v[kPoolUnroll];
#pragma unroll
    for (int u = 0; u < kPoolUnroll; ++u) v[u] = __ldg(src + (long)(r + u) * g.pitch);
#pragma unroll
    for (int u = 0; u < kPoolUnroll; ++u) {
      float f[8];
      unpack8(v[u], f);
#pragma unroll
      for (int j = 0; j < 8; ++j) s[j] += f[j];
    }
  }
  for (; r < g.R; ++r) {
    float f[8];
    unpack8(__ldg(src + (long)r * g.pitch), f);
#pragma unroll
    for (int j = 0; j < 8; ++j) s[j] += f[j];
  }
  float4* dst = reinterpret_cast<float4*>(pool + (((long)cand * kKC + kc) * g.P + pp) * 8);
  const float inv = 1.f / (float)g.R;
  dst[0] = make_float4(s[0] * inv, s[1] * inv, s[2] * inv, s[3] * inv);
  dst[1] = make_float4(s[4] * inv, s[5] * inv, s[6] * inv, s[7] * inv);
}

// ---- fused path: the stack kernel leaves the read-axis SUM of a segment's output as bf16 group sums (dan_stack.cuh: one group
// per (block of kStkBlockReads reads, slot), written by TMA bulk reductions). These kernels add the groups of a candidate in
// fp32, in a fixed order, and divide by the read count (AvgPool2d over all rows, empty ones included: model.py:194,304).
__device__ __forceinline__ void group_mean8(const uint4* __restrict__ sums, int cand, int kc, int pp, int P, int R, float (&s)[8]) {
  const int bpc = (R + kStkBlockReads - 1) / kStkBlockReads;
#pragma unroll
  for (int j = 0; j < 8; ++j) s[j] = 0.f;
  for (int b = 0; b < bpc; ++b) {
    const int nr = min(kStkBlockReads, R - b * kStkBlockReads);
    for (int sl = 0; sl < 2; ++sl) {
      if ((nr + 1 - sl) / 2 == 0) continue;                       // a block of one read has no slot-1 group
      float f[8];
      unpack8(__ldg(sums + (((long)cand * (2 * bpc) + 2 * b + sl) * kKC + kc) * P + pp), f);
#pragma unroll
      for (int j = 0; j < 8; ++j) s[j] += f[j];
    }
  }
  const float inv = 1.f / (float)R;
#pragma unroll
  for (int j = 0; j < 8; ++j) s[j] *= inv;
}

// read-mean of the layer in front of a pool-add (model.py:766-772) -> A operand of the pool-bias-map GEMM: row (cand*P + p'), columns
// tap*C + c holding bf16(pool[c][p' + (tap-1)*dil]) (zero outside the read: Conv2d zero padding, model.py:214-229)
__global__ void __launch_bounds__(64) pool_groups_im2col_kernel(const uint4* __restrict__ sums, int P, int R, uint4* __restrict__ im2col, int dil) {
  const int cand = blockIdx.y, kc = blockIdx.z;
  const int pp = blockIdx.x * blockDim.x + threadIdx.x;
  if (pp >= P) return;
  float s[8];
  group_mean8(sums, cand, kc, pp, P, R, s);
  const uint4 v = pack8(s);
  uint4* row0 = im2col + (long)cand * P * (3 * kKC) + kc;            // 3*kKC 16-byte pieces per row
#pragma unroll
  for (int tap = 0; tap < 3; ++tap) {
    const int pd = pp - (tap - 1) * dil;                             // the output position that reads this value through `tap`
    if (pd >= 0 && pd < P) row0[(long)pd * (3 * kKC) + tap * kKC] = v;
  }
  if (pp < dil) row0[(long)pp * (3 * kKC)] = make_uint4(0, 0, 0, 0);                        // tap 0 reaches in front of the read
  if (pp >= P - dil) row0[(long)pp * (3 * kKC) + 2 * kKC] = make_uint4(0, 0, 0, 0);         // tap 2 reaches behind it
}

// read-mean of the final layer (model.py:826) -> mean block of the pooled features; the max block next to it (model.py:825) is written
// by the stack kernel itself (bulk max-reductions) after fcin_max_init_kernel has set it to -inf. The pooled block is the head of the
// FC input, or a buffer of its own when the post-pool Linear follows (dan_bf16_forward).
__global__ void __launch_bounds__(64) fcin_mean_kernel(const uint4* __restrict__ sums, int P, int R, uint4* __restrict__ fcin, long fc_kstride, long mean_piece0, int cand0) {
  const int cand = blockIdx.y, kc = blockIdx.z;
  const int pp = blockIdx.x * blockDim.x + threadIdx.x;
  if (pp >= P) return;
  float s[8];
  group_mean8(sums, cand, kc, pp, P, R, s);
  fcin[(long)(cand0 + cand) * fc_kstride + mean_piece0 + (long)kc * P + pp] = pack8(s);
}
__global__ void fcin_max_init_kernel(uint4* __restrict__ fcin, long fc_kstride, int cand0, int cands, int pieces) {
  const long total = (long)cands * pieces;
  const uint4 ninf = make_uint4(0xFF80FF80u, 0xFF80FF80u, 0xFF80FF80u, 0xFF80FF80u);       // bf16 -inf
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x)
    fcin[(cand0 + i / pieces) * fc_kstride + i % pieces] = ninf;
}

// ---- pool bias map (fused stack path). The read-mean pool-add in front of a conv layer (model.py:734-742) is linear:
//   conv(x + pool) + b = conv(x) + [conv(pool) + b],
// and the bracket is the same for all reads of a candidate. It is computed once per candidate on the tensor cores (tma_gemm over the
// im2col rows above) and stored as bf16 pairs in exactly the order in which the stack kernel's epilogue threads hold the accumulator
// (tcgen05.ld 16x256b fragments, dan_stack_epi.cuh): per candidate 8 roles (position half h, lane quadrant q) x 7 chunks of 16
// positions x 32 lanes x 8 words; word gi*4 + j = channel 32q + 8j + lane/4, positions 8*(g0 + gi) + 2*(lane%4) + {0,1} with
// g0 = (h ? 14 : 0) + 2*chunk. The layer's epilogue adds it instead of the per-channel bias; the per-read pool-add (103 KB of L2
// reads and a 54 KB shared-memory read-modify-write on every read boundary) disappears.
__global__ void bmap_pack_kernel(const float* __restrict__ gmap, const float* __restrict__ bias, uint4* __restrict__ out, int cands, int P) {
  const long total = (long)cands * 8 * 7 * 32 * 2;
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int half = (int)(i & 1), lane = (int)((i >> 1) & 31);
    long t = i >> 6;
    const int chunk = (int)(t % 7); t /= 7;
    const int role = (int)(t % 8); const long cand = t / 8;
    const int h = role >> 2, q = role & 3, g0 = (h ? 14 : 0) + 2 * chunk, gi = half;
    uint32_t w[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int c = 32 * q + 8 * j + (lane >> 2), pos = 8 * (g0 + gi) + 2 * (lane & 3);
      const float b = bias[c];
      const float lo = pos < P ? gmap[(cand * P + pos) * kC + c] + b : 0.f;
      const float hi = pos + 1 < P ? gmap[(cand * P + pos + 1) * kC + c] + b : 0.f;
      w[j] = pack_bf16x2(lo, hi);
    }
    out[i] = make_uint4(w[0], w[1], w[2], w[3]);
  }
}

// out = bf16(h + pool) on data rows, 0 on gap rows   (model.py:742)
__global__ void add_pool_bf16_kernel(const uint4* __restrict__ h, const float* __restrict__ pool, uint4* __restrict__ out,
                                     long kstride, long rows, RowGeom g) {
  const long total = rows * kKC;
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int kc = (int)(i / rows); const long row = i - (long)kc * rows;
    const int pp = (int)(row % g.pitch); const long cand = row / ((long)g.R * g.pitch);
    uint4 v = h[kc * kstride + kLead + row];
    if (pp < g.P) {
      float f[8];
      unpack8(v, f);
      const float4* a = reinterpret_cast<const float4*>(pool + ((cand * kKC + kc) * g.P + pp) * 8);
      const float4 a0 = a[0], a1 = a[1];
      f[0] += a0.x; f[1] += a0.y; f[2] += a0.z; f[3] += a0.w; f[4] += a1.x; f[5] += a1.y; f[6] += a1.z; f[7] += a1.w;
      v = pack8(f);
    }
    out[kc * kstride + kLead + row] = v;
  }
}

// layer-wise fallback path: final max ‖ mean over reads -> pooled-feature pieces (bf16 feature order of both paths: max (c/8, p, c%8) | mean likewise)
__global__ void __launch_bounds__(64) pool_final_bf16_kernel(const uint4* __restrict__ h, long kstride, uint4* __restrict__ fcin, long fc_kstride,
                                       int cand0, RowGeom g, int skip_max) {
  const int cand = blockIdx.y, kc = blockIdx.z;
  const int pp = blockIdx.x * blockDim.x + threadIdx.x;
  if (pp >= g.P) return;
  float s[8] = {0, 0, 0, 0, 0, 0, 0, 0}, mx[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) mx[j] = -INFINITY;
  const uint4* src = h + kc * kstride + kLead + (long)cand * g.R * g.pitch + pp;
  int r = 0;
  for (; r + kPoolUnroll <= g.R; r += kPoolUnroll) {
    uint4 v[kPoolUnroll];
#pragma unroll
    for (int u = 0; u < kPoolUnroll; ++u) v[u] = __ldg(src + (long)(r + u) * g.pitch);
#pragma unroll
    for (int u = 0; u < kPoolUnroll; ++u) {
      float f[8];
      unpack8(v[u], f);
#pragma unroll
      for (int j = 0; j < 8; ++j) { s[j] += f[j]; mx[j] = fmaxf(mx[j], f[j]); }
    }
  }
  for (; r < g.R; ++r) {
    float f[8];
    unpack8(__ldg(src + (long)r * g.pitch), f);
#pragma unroll
    for (int j = 0; j < 8; ++j) { s[j] += f[j]; mx[j] = fmaxf(mx[j], f[j]); }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) s[j] /= (float)g.R;
  uint4* row = fcin + (long)(cand0 + cand) * fc_kstride;          // fc_kstride = pieces per row of the pooled-feature buffer
  if (skip_max) {
    row[(long)kc * g.P + pp] = pack8(s);
  } else {
    row[(long)kc * g.P + pp] = pack8(mx);
    row[(long)(kKC + kc) * g.P + pp] = pack8(s);
  }
}

// highway: hw fp32 partial [l][read][bott] + bias -> relu -> FC input pieces   (model.py:853-859)
__global__ void highway_finish_bf16_kernel(const float* __restrict__ hw, long layer_stride, const float* const* __restrict__ bias_by_layer,
                                           int L, int bott, int R, int concat, uint4* __restrict__ fcin, long fc_kstride,
                                           long base_kc, int cand0, int cands) {
  const int o8n = bott / 8;
  const long total = (long)cands * (concat ? L : 1) * R * o8n;
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int o8 = (int)(i % o8n); long t = i / o8n;
    const int r = (int)(t % R); t /= R;
    const int l = concat ? (int)(t % L) : 0; const long cand = concat ? t / L : t;
    float f[8];
    if (concat) {
      const float* src = hw + l * layer_stride + (cand * R + r) * bott + o8 * 8;
#pragma unroll
      for (int j = 0; j < 8; ++j) f[j] = fmaxf(src[j] + bias_by_layer[l][o8 * 8 + j], 0.f);
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) f[j] = 0.f;
      for (int k = 0; k < L; ++k) {
        const float* src = hw + k * layer_stride + (cand * R + r) * bott + o8 * 8;
#pragma unroll
        for (int j = 0; j < 8; ++j) f[j] += src[j] + bias_by_layer[k][o8 * 8 + j];
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) f[j] = fmaxf(f[j] / (float)L, 0.f);
    }
    fcin[(long)(cand0 + cand) * fc_kstride + base_kc + ((long)l * R + r) * o8n + o8] = pack8(f);
  }
}

// =====================================================================================================
// Weight packing (fp32 state_dict tensors -> bf16 operand images)
// =====================================================================================================
__device__ __forceinline__ void store_bf16(uint4* base, long piece, int j, float v) {
  reinterpret_cast<__nv_bfloat16*>(base + piece)[j] = __float2bfloat16_rn(v);
}
// conv (Cout, Cin, 1, 3) -> [tap][kc][n][8]
__global__ void pack_conv_bf16_kernel(const float* __restrict__ w, uint4* __restrict__ out, int Cin, int kc_in) {
  const long total = (long)3 * kc_in * kC * 8;
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int j = (int)(i & 7); long t = i >> 3;
    const int n = (int)(t % kC); t /= kC;
    const int kc = (int)(t % kc_in); const int tap = (int)(t / kc_in);
    const int c = kc * 8 + j;
    store_bf16(out, ((long)tap * kc_in + kc) * kC + n, j, c < Cin ? w[((long)n * Cin + c) * 3 + tap] : 0.f);
  }
}
// Feature order of the bf16 path's FC input (and of the post-pool Linear's input) against the reference's (model.py:833-859):
//   * pooled max | mean features: the kernels keep (block, c / 8, p, c % 8) — one 16-byte piece per (c / 8, p), the unit of the stack
//     kernel's bulk reductions — where the reference flattens (block, c, p);
//   * post-pool Linear outputs (pool_combine_dimension > 0): the reference's order;
//   * highway features: the kernels keep (layer, read, o), the reference (layer, o, read).
// Column k of such an input -> the reference's column. The leading `permuted` columns are pooled features, columns up to `hw_base` are
// in the reference's order, the rest is the highway block. Weight packers and the FC-input test hook both go through this map.
__device__ __forceinline__ long fc_ref_column(long k, long permuted, long hw_base, int P, int C, int R, int bott) {
  if (k < permuted) {
    const long blk = k / ((long)P * C);            // 0 = max block (or mean when skip_max), 1 = mean block
    const long rem = k - blk * P * C;
    const int kc8 = (int)(rem / (P * 8)), pp = (int)((rem / 8) % P), c = kc8 * 8 + (int)(rem % 8);
    return (blk * C + c) * (long)P + pp;
  }
  if (k < hw_base) return k;
  const long h = k - hw_base;
  const int o = (int)(h % bott); const long lr = h / bott;
  const int r = (int)(lr % R); const int l = (int)(lr / R);
  return hw_base + (long)l * bott * R + (long)o * R + r;
}
// where the blocks of the FC input sit: pooled features at the head (pool_combine_dimension 0), or the post-pool Linear's D outputs
struct FcInLayout { long permuted, hw_base; };
inline FcInLayout fc_in_layout(const dan_model* m) {
  const int D = m->cfg.pool_combine_dimension;
  return D > 0 ? FcInLayout{0, D} : FcInLayout{m->pooled, m->pooled};
}

// linear-like (N, K) fp32 with optional source-column map -> bf16 row-major [Npad][Kpad] (mode 3: UMMA chunk image [kc][Npad][8])
__global__ void pack_linear_bf16_kernel(const float* __restrict__ w, uint4* __restrict__ out, int N, int Npad, int K, int Kpad,
                                        int mode, int P, int C, int R, int bott, long permuted, long hw_base) {
  // mode 0: identity columns. mode 1: FC-input feature order (fc_ref_column). mode 2: compression (O, Cb, 1, P): k = ((c/8)*P + p)*8 + c%8
  // mode 4: conv weight (Cout, C, 1, 3) with k = tap*C + cin
  const long total = (long)(Kpad / 8) * Npad * 8;
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int j = (int)(i & 7); long t = i >> 3;
    const int n = (int)(t % Npad); const long kc = t / Npad;
    const long k = kc * 8 + j;
    float v = 0.f;
    if (n < N && k < K) {
      long src = k;
      if (mode == 1) {
        src = fc_ref_column(k, permuted, hw_base, P, C, R, bott);
      } else if (mode == 2) {                             // K order of the T matrix: (c / 8, p, c % 8)
        const int g = (int)(k / (P * 8)), rem = (int)(k % (P * 8));
        const int pp = rem / 8, c = g * 8 + rem % 8;
        src = (long)c * P + pp;                           // within row n: (c, p)
      } else if (mode == 4) {
        src = (k % C) * 3 + k / C;
      }
      v = w[(long)n * K + src];
    }
    if (mode == 3) store_bf16(out, kc * Npad + n, j, v);
    else reinterpret_cast<__nv_bfloat16*>(out)[(long)n * Kpad + k] = __float2bfloat16_rn(v);
  }
}

// per-layer epilogue constants [6][128]: conv bias | BN scale | BN shift | residual bias | -bias | scale * bias + shift (built on the
// device from the fp32 store; the last two are what the stack kernel's FMNMX + FFMA epilogue uses, dan_stack_epi.cuh)
constexpr int kChanRows = 6;
__global__ void chan_table_kernel(const float* __restrict__ bias, const float* __restrict__ scale, const float* __restrict__ shift,
                                  const float* __restrict__ rbias, float* __restrict__ out) {
  const int c = threadIdx.x;
  out[c] = bias[c];
  out[kC + c] = scale ? scale[c] : 1.f;
  out[2 * kC + c] = shift ? shift[c] : 0.f;
  out[3 * kC + c] = rbias ? rbias[c] : 0.f;
  out[4 * kC + c] = -bias[c];
  out[5 * kC + c] = fmaf(scale ? scale[c] : 1.f, bias[c], shift ? shift[c] : 0.f);
}

struct Bf16Weights {
  uint4* wconv[DAN_MAX_LAYERS]; uint4* wres[DAN_MAX_LAYERS]; uint4* wbott[DAN_MAX_LAYERS]; uint4* wcomp[DAN_MAX_LAYERS];
  uint4* wcomp_all;                   // all layers' compression weights, [L][bott][P*bott] bf16 (one batched GEMM operand)
  uint4* fcw[DAN_MAX_FC]; uint4* headw;
  uint4* postw;                       // post-pool Linear (pool_combine_dimension > 0): [D][pooledPad] bf16, columns in pooled-feature order
  uint4* wbmap[DAN_MAX_LAYERS];       // layers fed by a read-mean pool-add: conv weight as a row-major GEMM operand [cout][tap*C + cin] bf16 (pool bias map)
  const float** comp_bias_ptrs;       // device array of L pointers
  uint8_t* wstream[DAN_MAX_LAYERS];   // conv | residual | bottleneck operand images of a layer, contiguous (dan_stack.cuh); kWeightReplicas copies
  size_t wstream_bytes[DAN_MAX_LAYERS];   // bytes of one copy (256-byte multiple)
  float* chan_dev;                    // [L][6][128] epilogue constants (chan_table_kernel)
  uint4* enc_tab;                     // [P][10][3] pieces: bf16(E[tok] + pe[p]) (enc_table_kernel)
  int num_sms;
};

inline int grid_for(long total, int block = 256) {
  long g = (total + block - 1) / block;
  return (int)(g < 1 ? 1 : (g > 148 * 32 ? 148 * 32 : g));
}

// the shipped channel set (embed_dim 20, q-scores, strands, ref/var masks: 45 -> 48 channels): the fused kernel encodes it itself
inline bool stack_encodes(const dan_model* m) {
  return m->cfg.embed_dim == 20 && m->cfg.use_q_scores && m->cfg.use_strands && m->cfg.use_reads_ref_var_mask && m->CinPad == 48;
}
// configurations the fused stack kernel takes (everything else runs layer by layer, dan_layerwise.cuh)
inline bool stack_fused(const dan_model* m) {
  if (m->flags & DAN_FLAG_LAYERWISE) return false;
  if (m->P != 201 || m->geom.gap > kStkLead) return false;
  if (m->cfg.highway && m->bott != kStkBott) return false;
  int seg = 1;
  for (int l = 1; l < m->L; ++l) {
    if (m->cfg.pool_after[l - 1]) {
      if (m->cfg.is_residual[l]) return false;      // a residual layer fed by a pool-add needs the un-pooled input as residual (model.py:732 vs :742)
      seg = 0;
    }
    if (++seg > kStkMaxSeg) return false;
  }
  return true;
}
constexpr int kCompSplits = 4;
inline int sum_groups_per_cand(const dan_model* m) { return 2 * ((m->R + kStkBlockReads - 1) / kStkBlockReads); }

// workspace carve-up ---------------------------------------------------------------------------------------
struct Bf16Plan {
  int S, Bc, BcPad;
  long rows, rowsPad, kstride;       // per pass; kstride = rows per chunk plane
  long readsPad;
  long hw_layer_stride;
  long t_layer_pieces;               // uint4 pieces of one layer's T matrix
  int fcKC;                          // FC input pieces
  int poolKC;                        // pieces per row of the pooled-feature buffer (pool_combine_dimension > 0)
  size_t off_zero_begin, off_x0, off_h[3], off_zero_end, off_t, off_pool, off_sums, off_im2col, off_bmapg, off_bmap, off_hw, off_part, off_pooled, off_fcin, off_fcx[DAN_MAX_FC], total;
  int maxN;
};

Bf16Plan make_plan(const dan_model* m, int batch) {
  Bf16Plan pl{};
  pl.S = m->pass_candidates < batch ? m->pass_candidates : (batch > 0 ? batch : 1);
  const int fc_chunk = dan_bf16_fc_chunk(m);
  pl.Bc = batch < fc_chunk ? (batch > 0 ? batch : 1) : fc_chunk;
  pl.BcPad = round_up_i(pl.Bc, 128);
  pl.rows = m->geom.rows_of(pl.S);
  pl.rowsPad = (pl.rows + 127) / 128 * 128;
  pl.kstride = kLead + pl.rowsPad + 8;
  pl.readsPad = ((long)pl.S * m->R + 127) / 128 * 128;
  pl.fcKC = m->fcInPad / 8;
  const bool fused = stack_fused(m);
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off += round_up_z(bytes, 1024); return o; };
  pl.off_zero_begin = off;
  pl.off_x0 = take(fused && stack_encodes(m) ? 0 : (size_t)(m->CinPad / 8) * pl.kstride * 16);
  for (int i = 0; i < 3; ++i) pl.off_h[i] = take(fused && i == 2 ? 0 : (size_t)kKC * pl.kstride * 16);     // fused: segments ping-pong; layer-wise: input, pool-added input, output
  pl.off_zero_end = off;
  const int bott = m->bott > 0 ? m->bott : 32;
  pl.t_layer_pieces = (long)m->P * (bott / 8) * pl.readsPad;
  pl.off_t = take((size_t)m->L * pl.t_layer_pieces * 16);
  pl.off_pool = take(fused ? 0 : (size_t)pl.S * m->P * kC * 4);
  pl.off_sums = take(fused ? (size_t)pl.S * sum_groups_per_cand(m) * kKC * m->P * 16 : 0);     // read-axis sum groups of the segment that just ran
  pl.off_im2col = take((size_t)pl.S * m->P * 3 * kC * 2);      // pool bias map (see bmap_pack_kernel): im2col of the read-mean, bf16 [cand*P + p][tap*C + c]
  pl.off_bmapg = take((size_t)pl.S * m->P * kC * 4);          // conv(pool), fp32 [cand*P + p][cout]
  pl.off_bmap = take((size_t)pl.S * kBmapBytesPerCand);      // conv(pool) + bias in the stack epilogue's fragment order, bf16 pairs
  pl.hw_layer_stride = pl.readsPad * bott;
  pl.off_hw = take((size_t)m->L * pl.hw_layer_stride * 4);
  pl.off_part = take((size_t)kCompSplits * m->L * pl.readsPad * bott * 4);     // split-K partials of the compression GEMM
  // with the post-pool Linear (model.py:841-843) the pooled max | mean block (wider than the FC input) is its own GEMM operand
  pl.poolKC = m->pooledPad / 8;
  pl.off_pooled = take(m->cfg.pool_combine_dimension > 0 ? (size_t)pl.poolKC * pl.BcPad * 16 : 0);     // [BcPad][pooledPad] bf16
  pl.off_fcin = take((size_t)pl.fcKC * pl.BcPad * 16);           // [BcPad][fcInPad] bf16, row-major
  pl.maxN = DAN_HEAD_PAD;
  for (int i = 0; i < m->cfg.num_fc; ++i) {
    pl.off_fcx[i] = take((size_t)(m->cfg.fc_sizes[i] / 8) * pl.BcPad * 16);
    if (m->cfg.fc_sizes[i] > pl.maxN) pl.maxN = m->cfg.fc_sizes[i];
  }
  pl.total = off;
  return pl;
}

}  // namespace

// ----------------------------------------------------------------------------------------------------------
const char* dan_bf16_unsupported_reason(const dan_model* m) {
  if (m->C != kC) return "the bf16 kernels are built for 128 conv channels";
  // N of the post-pool GEMM and of the FC trunk's GEMMs is cut into 32- or 64-wide tiles (run_gemm2)
  if (m->cfg.pool_combine_dimension % 32) return "pool_combine_dimension must be a multiple of 32";
  if (m->cfg.highway && !(m->bott == 32 || m->bott == 64)) return "the highway bottleneck must be 32 or 64 wide";
  if (m->geom.gap > kLead) return "dilation above 8";
  if (m->CinPad % 16) return "padded input channels must be a multiple of 16";
  // a layer-1 input tile slot (dan_layerwise.cuh) and the fused kernel's read buffer (kStkBuf) hold kKC = 16 channel planes
  if (m->CinPad > kC) return "more than 128 padded input channels (embed_dim 62-64 with q-scores, strands and masks)";
  for (int i = 0; i < m->cfg.num_fc; ++i) if (m->cfg.fc_sizes[i] % 32) return "FC widths must be multiples of 32";
  return nullptr;
}
int dan_bf16_supported(const dan_model* m) { return dan_bf16_unsupported_reason(m) == nullptr; }
int dan_bf16_route(const dan_model* m) { return dan_bf16_unsupported_reason(m) ? 0 : stack_fused(m) ? 1 : 2; }

size_t dan_bf16_workspace_bytes(const dan_model* m, int batch) {
  if (const char* why = dan_bf16_unsupported_reason(m)) {
    dan_set_error("bf16 tcgen05 path does not cover this configuration: %s", why);
    return 0;
  }
  return make_plan(m, batch).total;
}

int dan_bf16_pack(dan_model* m, const dan_weights* w, cudaStream_t st) {
  Bf16Weights* bw = static_cast<Bf16Weights*>(m->bf16_store);
  if (!bw) {
    bw = new Bf16Weights();
    memset(bw, 0, sizeof(*bw));
    m->bf16_store = bw;
    cudaDeviceGetAttribute(&bw->num_sms, cudaDevAttrMultiProcessorCount, m->device);
  }
  const int L = m->L, bott = m->bott, P = m->P, R = m->R;
  auto alloc = [&](uint4** p, size_t pieces) -> int {
    if (*p) return DAN_OK;
    DAN_CUDA_TRY(cudaMalloc(p, pieces * 16));
    return DAN_OK;
  };
  int rc;
  if (!bw->chan_dev) DAN_CUDA_TRY(cudaMalloc(&bw->chan_dev, sizeof(float) * DAN_MAX_LAYERS * kChanRows * kC));
  for (int l = 0; l < L; ++l) {
    const int cin = l == 0 ? m->Cin : kC, kc_in = (l == 0 ? m->CinPad : kC) / 8;
    if (!bw->wstream[l]) {
      const size_t conv_b = (size_t)3 * kc_in * kC * 16, res_b = m->cfg.is_residual[l] ? (size_t)kKC * kC * 16 : 0, bott_b = m->cfg.highway ? (size_t)kKC * bott * 16 : 0;
      bw->wstream_bytes[l] = round_up_z(conv_b + res_b + bott_b, 256);
      DAN_CUDA_TRY(cudaMalloc(&bw->wstream[l], bw->wstream_bytes[l] * kWeightReplicas));
      bw->wconv[l] = reinterpret_cast<uint4*>(bw->wstream[l]);
      if (res_b) bw->wres[l] = reinterpret_cast<uint4*>(bw->wstream[l] + conv_b);
      if (bott_b) bw->wbott[l] = reinterpret_cast<uint4*>(bw->wstream[l] + conv_b + res_b);
    }
    pack_conv_bf16_kernel<<<grid_for((long)3 * kc_in * kC * 8), 256, 0, st>>>(w->conv_w[l], bw->wconv[l], cin, kc_in);
    if (l > 0 && m->cfg.pool_after[l - 1]) {
      if ((rc = alloc(&bw->wbmap[l], (size_t)kC * 3 * kC / 8))) return rc;
      pack_linear_bf16_kernel<<<grid_for((long)3 * kC * kC), 256, 0, st>>>(w->conv_w[l], bw->wbmap[l], kC, kC, 3 * kC, 3 * kC, 4, P, kC, R, bott, 0, 0);
    }
    if (m->cfg.is_residual[l]) {
      pack_linear_bf16_kernel<<<grid_for((long)kKC * kC * 8), 256, 0, st>>>(w->res_w[l], bw->wres[l], kC, kC, kC, kC, 3, P, kC, R, bott, 0, 0);
    }
    if (m->cfg.highway) {
      pack_linear_bf16_kernel<<<grid_for((long)kKC * bott * 8), 256, 0, st>>>(w->bott_w[l], bw->wbott[l], bott, bott, kC, kC, 3, P, kC, R, bott, 0, 0);
      const int K = P * bott;
      if ((rc = alloc(&bw->wcomp_all, (size_t)L * (K / 8) * bott))) return rc;
      bw->wcomp[l] = bw->wcomp_all + (size_t)l * (K / 8) * bott;
      pack_linear_bf16_kernel<<<grid_for((long)K * bott), 256, 0, st>>>(w->comp_w[l], bw->wcomp[l], bott, bott, K, K, 2, P, kC, R, bott, 0, 0);
    }
    // epilogue constants (the fp32 packer already folded BatchNorm on this stream)
    chan_table_kernel<<<1, kC, 0, st>>>(m->convB[l], m->cfg.use_batchnorm ? m->bnScale[l] : nullptr, m->cfg.use_batchnorm ? m->bnShift[l] : nullptr,
                                        m->cfg.is_residual[l] ? m->resB[l] : nullptr, bw->chan_dev + (size_t)l * kChanRows * kC);
  }
  const int D = m->cfg.pool_combine_dimension;
  if (D > 0) {      // post_pool_conv1D (D, pooled): its input columns are the pooled features in the kernels' order
    if ((rc = alloc(&bw->postw, (size_t)(m->pooledPad / 8) * D))) return rc;
    pack_linear_bf16_kernel<<<grid_for((long)m->pooledPad * D), 256, 0, st>>>(w->post_pool_w, bw->postw, D, D, m->pooled, m->pooledPad, 1, P, kC, R, bott,
                                                                              m->pooled, m->pooled);
  }
  const FcInLayout fl = fc_in_layout(m);
  int K = m->fcIn, Kpad = m->fcInPad;
  for (int i = 0; i < m->cfg.num_fc; ++i) {
    const int N = m->cfg.fc_sizes[i];
    if ((rc = alloc(&bw->fcw[i], (size_t)(Kpad / 8) * N))) return rc;
    pack_linear_bf16_kernel<<<grid_for((long)Kpad * N), 256, 0, st>>>(w->fc_w[i], bw->fcw[i], N, N, K, Kpad, i == 0 ? 1 : 0, P, kC, R, bott,
                                                                      fl.permuted, fl.hw_base);
    K = N; Kpad = N;
  }
  if ((rc = alloc(&bw->headw, (size_t)(m->hidden / 8) * DAN_HEAD_PAD))) return rc;
  pack_linear_bf16_kernel<<<grid_for((long)m->hidden * DAN_HEAD_PAD), 256, 0, st>>>(w->head_w, bw->headw, DAN_NUM_HEAD_OUTPUTS, DAN_HEAD_PAD, m->hidden, m->hidden, 0, P, kC, R, bott, 0, 0);
  for (int l = 0; l < L; ++l)
    for (int r = 1; r < kWeightReplicas; ++r)
      DAN_CUDA_TRY(cudaMemcpyAsync(bw->wstream[l] + (size_t)r * bw->wstream_bytes[l], bw->wstream[l], bw->wstream_bytes[l], cudaMemcpyDeviceToDevice, st));
  if (stack_encodes(m)) {
    if ((rc = alloc(&bw->enc_tab, (size_t)P * DAN_VOCAB * 3))) return rc;
    enc_table_kernel<<<grid_for((long)P * DAN_VOCAB * 24), 256, 0, st>>>(m->emb, m->pe, P, m->cfg.embed_dim, bw->enc_tab);
  }
  if (m->cfg.highway) {
    // device array of the compression-bias pointers, filled from pinned-free host memory through the stream (small, ordered with the kernels)
    if (!bw->comp_bias_ptrs) DAN_CUDA_TRY(cudaMalloc(&bw->comp_bias_ptrs, sizeof(float*) * DAN_MAX_LAYERS));
    DAN_CUDA_TRY(cudaMemcpyAsync(bw->comp_bias_ptrs, m->compB, sizeof(float*) * L, cudaMemcpyHostToDevice, st));
  }
  DAN_CUDA_TRY(cudaGetLastError());
  return DAN_OK;
}

void dan_bf16_free(dan_model* m) {
  Bf16Weights* bw = static_cast<Bf16Weights*>(m->bf16_store);
  if (!bw) return;
  for (int l = 0; l < DAN_MAX_LAYERS; ++l) { cudaFree(bw->wstream[l]); cudaFree(bw->wbmap[l]); }
  cudaFree(bw->wcomp_all);
  cudaFree(bw->chan_dev);
  cudaFree(bw->enc_tab);
  for (int i = 0; i < DAN_MAX_FC; ++i) cudaFree(bw->fcw[i]);
  cudaFree(bw->headw);
  cudaFree(bw->postw);
  cudaFree(bw->comp_bias_ptrs);
  delete bw;
  m->bf16_store = nullptr;
}

int dan_bf16_forward(dan_model* m, const DevInputs& in, int batch, float* heads_out, void* ws, size_t ws_bytes, cudaStream_t st) {
  Bf16Weights* bw = static_cast<Bf16Weights*>(m->bf16_store);
  if (!bw) { dan_set_error("bf16 weights not packed"); return DAN_E_INVALID; }
  const Bf16Plan pl = make_plan(m, batch);
  if (ws_bytes < pl.total) { dan_set_error("workspace too small: %zu < %zu", ws_bytes, pl.total); return DAN_E_WORKSPACE; }
  char* base = static_cast<char*>(ws);
  const RowGeom g = m->geom;
  const int L = m->L, bott = m->bott, P = m->P, R = m->R;
  uint4* X0 = reinterpret_cast<uint4*>(base + pl.off_x0);
  uint4* H[3]; for (int i = 0; i < 3; ++i) H[i] = reinterpret_cast<uint4*>(base + pl.off_h[i]);
  uint4* T = reinterpret_cast<uint4*>(base + pl.off_t);
  float* POOL = reinterpret_cast<float*>(base + pl.off_pool);
  uint4* SUMS = reinterpret_cast<uint4*>(base + pl.off_sums);
  uint4* IM2COL = reinterpret_cast<uint4*>(base + pl.off_im2col);
  float* BMAPG = reinterpret_cast<float*>(base + pl.off_bmapg);
  uint4* BMAP = reinterpret_cast<uint4*>(base + pl.off_bmap);
  float* HW = reinterpret_cast<float*>(base + pl.off_hw);
  uint4* FCIN = reinterpret_cast<uint4*>(base + pl.off_fcin);
  const int D = m->cfg.pool_combine_dimension;
  // pooled max | mean pieces: the head of the FC input, or (post-pool Linear, model.py:841-843) the A operand of the post-pool GEMM
  uint4* POOLED = D > 0 ? reinterpret_cast<uint4*>(base + pl.off_pooled) : FCIN;
  const long pool_kstride = D > 0 ? pl.poolKC : pl.fcKC;
  const FcInLayout fl = fc_in_layout(m);
  const bool fused = stack_fused(m);
  const bool enc_in_kernel = fused && stack_encodes(m) && bw->enc_tab != nullptr;
  const long mean_piece0 = m->cfg.skip_final_maxpool ? 0 : (long)kKC * P;      // pooled pieces: max block | mean block
  // highway compression (model.py:776) of every layer of a pass as ONE batched GEMM: HW[l][read][o] = T[l][read][:] . Wc[l][o][:]
  auto run_compression = [&](int l0, int nl, int reads) -> int {
    const long K = (long)P * bott;
    Gemm2Operand A{T + (long)l0 * pl.t_layer_pieces, reads, K * 2, pl.t_layer_pieces * 16};
    Gemm2Operand B{bw->wcomp[l0], bott, K * 2, K * 2 * bott};
    Gemm2Params gp{};
    gp.M = reads; gp.N = bott; gp.K = (int)K; gp.mode = kG2Raw;
    gp.part = reinterpret_cast<float*>(base + pl.off_part); gp.splits = kCompSplits;      // K = 6432 in 4 fixed ranges: same sums for every batch shape, 4x the CTAs
    gp.out = HW + (long)l0 * pl.hw_layer_stride; gp.out_batch_stride = pl.hw_layer_stride; gp.ldo = bott;
    return run_gemm2(A, B, gp, nl, bw->num_sms, st);
  };
  int rc;

  static DanSmemAttr enc_attr, layer_attr, stack_attr;
  const size_t enc_smem = encode_smem_bytes(P, R, m->cfg.embed_dim);
  if (!enc_in_kernel) DAN_CUDA_TRY(enc_attr.ensure(encode_rows_bf16_kernel, enc_smem));
  if (fused) DAN_CUDA_TRY(stack_attr.ensure(dan_stack_kernel, kStkSmemBytes));
  else DAN_CUDA_TRY(layer_attr.ensure(dan_layer_kernel, 227 * 1024));
  // layer-wise path: halo rows (and the rows past the last tile) must read as zero: clear the row matrices once per call.
  // The fused path loads and stores exactly the P data rows of every read and keeps its zero rows in shared memory.
  if (!fused) DAN_CUDA_TRY(cudaMemsetAsync(base + pl.off_zero_begin, 0, pl.off_zero_end - pl.off_zero_begin, st));

  // one persistent launch of dan_stack_kernel over layers [l, l_end) of a pass (dan_stack.cuh)
  auto launch_segment = [&](int l, int l_end, long cand0, const uint4* seg_in, uint4* seg_out, bool with_bmap, bool want_sums, bool final_seg, int s0, int ns) -> int {
    StackParams sp{};
    if (l == 0 && enc_in_kernel) { sp.in_mode = kStkInEncode; sp.bytes = in; sp.cand0 = cand0; sp.enc_tab = bw->enc_tab; }
    else { sp.in_mode = kStkInPlanes; sp.in = seg_in; sp.in_kstride = pl.kstride; }
    sp.out = seg_out; sp.out_kstride = pl.kstride;
    if (want_sums || final_seg) { sp.sums = SUMS; sp.groups_per_cand = sum_groups_per_cand(m); }
    if (final_seg && !m->cfg.skip_final_maxpool) { sp.maxv = POOLED + (long)s0 * pool_kstride; sp.max_stride = pool_kstride; }
    sp.bmap = with_bmap ? BMAP : nullptr;
    sp.cands = ns; sp.R = R; sp.P = P; sp.pitch = g.pitch; sp.highway = m->cfg.highway; sp.num_layers = l_end - l;
    for (int k = l; k < l_end; ++k) {
      StackLayer& SL = sp.layer[k - l];
      SL.wstream = bw->wstream[k]; SL.wreplica_stride = bw->wstream_bytes[k]; SL.chan = bw->chan_dev + (size_t)k * kChanRows * kC; SL.bbias = m->bottB[k];
      SL.tout = T + (long)k * pl.t_layer_pieces;
      SL.kc_in = (k == 0 ? m->CinPad : kC) / 8; SL.conv_blocks = 3 * SL.kc_in / 2;
      SL.dil = m->cfg.dilation[k]; SL.residual = m->cfg.is_residual[k];
    }
    const int blocks = ns * (sum_groups_per_cand(m) / 2);
    const int grid = blocks < bw->num_sms ? blocks : bw->num_sms;
#ifdef DAN_STK_PROF
    const size_t prof_words = (size_t)64 * grid + 4 * kStkTraceCap;
    DAN_CUDA_TRY(cudaMalloc(&sp.prof, sizeof(unsigned long long) * prof_words));
    DAN_CUDA_TRY(cudaMemsetAsync(sp.prof, 0, sizeof(unsigned long long) * prof_words, st));
#endif
    { DanProfScope ps(DAN_PROF_CONV_STACK, st); dan_stack_kernel<<<grid, kStkThreads, kStkSmemBytes, st>>>(sp); }
    dan_count_launch();
    DAN_CUDA_TRY(cudaGetLastError());
#ifdef DAN_STK_PROF
    {   // development build (python -m dl4vc_b200.build --prof): per-role cycle counters, mean over CTAs, one line per launch
      std::vector<unsigned long long> hbuf(prof_words);
      DAN_CUDA_TRY(cudaStreamSynchronize(st));
      DAN_CUDA_TRY(cudaMemcpy(hbuf.data(), sp.prof, hbuf.size() * 8, cudaMemcpyDeviceToHost));
      cudaFree(sp.prof);
      double a[64] = {0};
      for (int c = 0; c < grid; ++c) for (int k = 0; k < 64; ++k) a[k] += (double)hbuf[c * 64 + k] / grid;
      const double reads = (double)ns * R / grid / 2;      // reads per slot
      fprintf(stderr, "[stkprof] layers %d-%d, %.0f reads/slot; cycles per read:", l + 1, l_end, reads);
      for (int sl = 0; sl < 2; ++sl)
        fprintf(stderr, " | issuer%d other %.0f wfull %.0f lag %.0f act_ready %.0f in_full %.0f bott_free %.0f total %.0f", sl, a[14 * sl] / reads, a[14 * sl + 1] / reads,
                a[14 * sl + 2] / reads, a[14 * sl + 3] / reads, a[14 * sl + 4] / reads, a[14 * sl + 5] / reads, a[14 * sl + 9] / reads);
      fprintf(stderr, "\n");
      for (int sl = 0; sl < 2; ++sl) {
        const double* e = a + 28 + 14 * sl;
        fprintf(stderr, "[stkprof]   epilogue slot %d: other %.0f wait-bott %.0f bott-epi %.0f wait-acc %.0f main-epi %.0f post-epi %.0f tma: bar %.0f wait0 %.0f issue %.0f | wait-read-out %.0f prepare %.0f arrive %.0f total %.0f\n", sl,
                e[0] / reads, e[1] / reads, e[2] / reads, e[3] / reads, e[4] / reads, e[5] / reads, e[10] / reads, e[11] / reads, e[6] / reads, e[7] / reads, e[8] / reads, e[12] / reads, e[9] / reads);
      }
      // event trace of CTA 0 (reads 10-13 of each slot): one file per segment shape, written once
      static int dumped[2] = {0, 0};
      if (!dumped[l > 0]) {
        dumped[l > 0] = 1;
        char path[128];
        snprintf(path, sizeof(path), "gpurun_out/stk_trace_l%d.txt", l + 1);
        if (FILE* f = fopen(path, "w")) {
          static const char* role[4] = {"issuer0", "issuer1", "epi0", "epi1"};
          for (int r = 0; r < 4; ++r)
            for (int i = 0; i < kStkTraceCap; ++i) {
              const unsigned long long v = hbuf[(size_t)64 * grid + (size_t)r * kStkTraceCap + i];
              if (v) fprintf(f, "%s %llu %llu\n", role[r], v >> 48, v & ((1ull << 48) - 1));
            }
          fclose(f);
        }
      }
    }
#endif
    return DAN_OK;
  };

  EncodeParams ep{};
  ep.in = in; ep.emb = m->emb; ep.pe = m->pe; ep.D = m->cfg.embed_dim; ep.Cin = m->Cin; ep.CinPad = m->CinPad;
  ep.use_q = m->cfg.use_q_scores; ep.use_s = m->cfg.use_strands; ep.use_m = m->cfg.use_reads_ref_var_mask; ep.g = g;

  for (int c0 = 0; c0 < batch; c0 += pl.Bc) {
    const int nb = batch - c0 < pl.Bc ? batch - c0 : pl.Bc;
    if (m->fcInPad != m->fcIn) DAN_CUDA_TRY(cudaMemsetAsync(FCIN, 0, (size_t)pl.fcKC * pl.BcPad * 16, st));
    for (int s0 = 0; s0 < nb; s0 += pl.S) {
      const int ns = nb - s0 < pl.S ? nb - s0 : pl.S;
      const long rows = g.rows_of(ns);
      const int num_tiles = (int)((rows + 127) / 128);
      if (!enc_in_kernel) {
        DanProfScope ps(DAN_PROF_ENCODE, st);
        encode_rows_bf16_kernel<<<ns, 256, enc_smem, st>>>(ep, (long)c0 + s0, X0, pl.kstride);
        dan_count_launch();
        DAN_CUDA_TRY(cudaGetLastError());
      }
      const uint4* cur = X0;
      int hsel = 0;
      if (fused) {
        // ---- fused path: one persistent launch per segment of layers without a pool-add in between (dan_stack.cuh) ----
        int l = 0;
        bool with_bmap = false;
        while (l < L) {
          int l_end = l + 1;
          while (l_end < L && !m->cfg.pool_after[l_end - 1]) ++l_end;
          const bool final_seg = l_end == L;
          const bool pool_next = !final_seg;             // segments end where a read-mean pool-add follows (or at the last layer)
          uint4* next = final_seg ? nullptr : H[hsel ^ 1];
          if (final_seg && !m->cfg.skip_final_maxpool) {
            { DanProfScope ps(DAN_PROF_POOL, st); fcin_max_init_kernel<<<grid_for((long)ns * kKC * P), 256, 0, st>>>(POOLED, pool_kstride, s0, ns, kKC * P); }
            dan_count_launch();
          }
          if ((rc = launch_segment(l, l_end, (long)c0 + s0, cur, next, with_bmap, pool_next, final_seg, s0, ns))) return rc;
          if (pool_next) {
            // bias map of layer l_end: read-mean of this segment's output (from the sum groups) -> conv(pool) on the tensor cores (rows =
            // candidate positions, K = 3 taps x 128 channels) -> + bias, in the stack epilogue's fragment order
            { DanProfScope ps(DAN_PROF_POOL, st); pool_groups_im2col_kernel<<<dim3((P + 63) / 64, ns, kKC), 64, 0, st>>>(SUMS, P, R, IM2COL, m->cfg.dilation[l_end]); }
            dan_count_launch();
            Gemm2Operand A{IM2COL, (long)ns * P, 3L * kC * 2, 0};
            Gemm2Operand B{bw->wbmap[l_end], kC, 3L * kC * 2, 0};
            Gemm2Params gp{};
            gp.M = ns * P; gp.N = kC; gp.K = 3 * kC; gp.mode = kG2Raw; gp.out = BMAPG; gp.out_batch_stride = 0; gp.ldo = kC;
            if ((rc = run_gemm2(A, B, gp, 1, bw->num_sms, st))) return rc;
            { DanProfScope ps(DAN_PROF_POOL, st); bmap_pack_kernel<<<grid_for((long)ns * kStkBmapPerCand), 256, 0, st>>>(BMAPG, m->convB[l_end], BMAP, ns, P); }
            dan_count_launch();
            DAN_CUDA_TRY(cudaGetLastError());
            with_bmap = true;
            cur = next; hsel ^= 1;
          } else {
            { DanProfScope ps(DAN_PROF_POOL, st); fcin_mean_kernel<<<dim3((P + 63) / 64, ns, kKC), 64, 0, st>>>(SUMS, P, R, POOLED, pool_kstride, mean_piece0, s0); }
            dan_count_launch();
            DAN_CUDA_TRY(cudaGetLastError());
          }
          l = l_end;
        }
        if (m->cfg.highway) {
          if ((rc = run_compression(0, L, ns * R))) return rc;
        }
      } else {
        for (int l = 0; l < L; ++l) {
          const uint4* conv_in = cur;
          if (l > 0 && m->cfg.pool_after[l - 1]) {
            uint4* hp = H[(hsel + 2) % 3];
            { DanProfScope ps(DAN_PROF_POOL, st); add_pool_bf16_kernel<<<grid_for(rows * kKC), 256, 0, st>>>(cur, POOL, hp, pl.kstride, rows, g); }
            dan_count_launch();
            DAN_CUDA_TRY(cudaGetLastError());
            conv_in = hp;
          }
          uint4* next = H[(hsel + 1) % 3];
          LayerParams lp{};
          lp.in = conv_in; lp.in_kstride = pl.kstride; lp.out = next; lp.out_kstride = pl.kstride;
          lp.tout = T + (long)l * pl.t_layer_pieces; lp.t_reads_stride = pl.readsPad;
          lp.resid = (m->cfg.is_residual[l] && conv_in != cur) ? cur : nullptr;   // residual excludes the pool term (model.py:732 vs :742)
          lp.wconv = bw->wconv[l]; lp.wres = bw->wres[l]; lp.wbott = bw->wbott[l];
          lp.rows_total = rows; lp.num_tiles = num_tiles; lp.pitch = g.pitch; lp.P = P; lp.gap = g.gap; lp.dil = m->cfg.dilation[l];
          lp.kc_in = (l == 0 ? m->CinPad : kC) / 8; lp.residual = m->cfg.is_residual[l]; lp.highway = m->cfg.highway; lp.bott = bott;
          lp.chan = bw->chan_dev + (size_t)l * kChanRows * kC; lp.bbias = m->bottB[l];
          const size_t smem = layer_smem_bytes(lp.kc_in, lp.residual, lp.highway, bott, g.gap);
          int grid = (num_tiles + kSlots - 1) / kSlots;
          if (grid > bw->num_sms) grid = bw->num_sms;
          { DanProfScope ps(DAN_PROF_CONV_STACK, st); dan_layer_kernel<<<grid, kLayerThreads, smem, st>>>(lp); }
          dan_count_launch();
          DAN_CUDA_TRY(cudaGetLastError());
          if (m->cfg.pool_after[l]) {
            { DanProfScope ps(DAN_PROF_POOL, st); pool_mean_bf16_kernel<<<dim3((P + 63) / 64, ns, kKC), 64, 0, st>>>(next, pl.kstride, POOL, g); }
            dan_count_launch();
            DAN_CUDA_TRY(cudaGetLastError());
          }
          if (m->cfg.highway) {
            if ((rc = run_compression(l, 1, ns * R))) return rc;
          }
          cur = next; hsel = (hsel + 1) % 3;
        }
        { DanProfScope ps(DAN_PROF_POOL, st); pool_final_bf16_kernel<<<dim3((P + 63) / 64, ns, kKC), 64, 0, st>>>(cur, pl.kstride, POOLED, pool_kstride, s0, g, m->cfg.skip_final_maxpool); }
        dan_count_launch();
        DAN_CUDA_TRY(cudaGetLastError());
      }
      if (m->cfg.highway) {
        const int Lh = m->cfg.concat_hw_reads ? L : 1;
        { DanProfScope ps(DAN_PROF_POOL, st); highway_finish_bf16_kernel<<<grid_for((long)ns * Lh * R * (bott / 8)), 256, 0, st>>>(
            HW, pl.hw_layer_stride, bw->comp_bias_ptrs, L, bott, R, m->cfg.concat_hw_reads, FCIN, pl.fcKC, fl.hw_base / 8, s0, ns); }
        dan_count_launch();
        DAN_CUDA_TRY(cudaGetLastError());
      }
    }
    if (D > 0) {
      // ---- post_pool_conv1D + ReLU (model.py:841-843) -> FC-input columns [0, D). One K = pooled contraction per row, unsplit: a row's
      // sum runs in the same order whatever the batch shape ----
      Gemm2Operand A{POOLED, nb, (long)pl.poolKC * 16, 0};
      Gemm2Operand B{bw->postw, D, (long)pl.poolKC * 16, 0};
      Gemm2Params gp{};
      gp.M = nb; gp.N = D; gp.K = m->pooled; gp.mode = kG2BiasReluBf16; gp.bias = m->postB;
      gp.out_bf16 = reinterpret_cast<__nv_bfloat16*>(FCIN); gp.ld_bf16 = m->fcInPad;
      if ((rc = run_gemm2(A, B, gp, 1, bw->num_sms, st))) return rc;
    }
    // ---- FC trunk + heads (model.py:917-958) ----
    const uint4* x = FCIN; int K = m->fcInPad;
    for (int i = 0; i < m->cfg.num_fc; ++i) {
      const int N = m->cfg.fc_sizes[i];
      uint4* y = reinterpret_cast<uint4*>(base + pl.off_fcx[i]);
      Gemm2Operand A{x, nb, (long)K * 2, 0};
      Gemm2Operand B{bw->fcw[i], N, (long)K * 2, 0};
      Gemm2Params gp{};
      gp.M = nb; gp.N = N; gp.K = K; gp.mode = kG2BiasReluBf16; gp.bias = m->fcB[i];
      gp.out_bf16 = reinterpret_cast<__nv_bfloat16*>(y); gp.ld_bf16 = N;
      if ((rc = run_gemm2(A, B, gp, 1, bw->num_sms, st))) return rc;
      x = y; K = N;
    }
    {
      Gemm2Operand A{x, nb, (long)K * 2, 0};
      Gemm2Operand B{bw->headw, DAN_HEAD_PAD, (long)K * 2, 0};
      Gemm2Params gp{};
      gp.M = nb; gp.N = DAN_HEAD_PAD; gp.K = K; gp.mode = kG2Heads; gp.bias = m->headB;
      gp.out = heads_out + (long)c0 * DAN_NUM_HEAD_OUTPUTS;
      if ((rc = run_gemm2(A, B, gp, 1, bw->num_sms, st))) return rc;
    }
  }
  return DAN_OK;
}

// ---- test hook for the bit-exact encoding work: the fused kernel's encoder prologue (stk_enc_fetch / stk_enc_rows / stk_enc_store, dan_stack.cuh)
// run stand-alone, one CTA per read, its six input planes written out in the reference's logical order (B, Cin, R, P) as fp32
namespace {
__global__ void __launch_bounds__(kStkEpiThreads) stack_encode_dump_kernel(StackParams p, int Cin, float* __restrict__ out) {
  __shared__ __align__(16) uint8_t buf[6 * kStkPlane];
  const int r = blockIdx.x, pos = threadIdx.x;
  const long cand = blockIdx.y;
  const StkEncBytes eb = stk_enc_fetch(p, cand, r, pos);
  const StkEncRows rows = stk_enc_rows(p, pos, 0, eb, stk_enc_fetch_cand(p, cand, pos));
  stk_enc_store(p, pos, eb, rows, buf);
  __syncthreads();
  for (int i = threadIdx.x; i < Cin * p.P; i += blockDim.x) {
    const int c = i / p.P, pp = i - c * p.P;
    const __nv_bfloat16 v = reinterpret_cast<const __nv_bfloat16*>(buf + (size_t)(c / 8) * kStkPlane + (size_t)(kStkLead + pp) * 16)[c % 8];
    out[((cand * Cin + c) * p.R + r) * p.P + pp] = __bfloat162float(v);
  }
}
}  // namespace

int dan_bf16_encode_reference_order(dan_model* m, const DevInputs& in, int batch, float* x0_out, cudaStream_t st) {
  Bf16Weights* bw = static_cast<Bf16Weights*>(m->bf16_store);
  if (!bw || !bw->enc_tab || !stack_encodes(m) || m->P > kStkN) { dan_set_error("the fused encoder prologue covers the shipped channel set only (embed_dim 20, q-scores, strands, ref/var masks)"); return DAN_E_UNSUPPORTED; }
  StackParams sp{};
  sp.in_mode = kStkInEncode; sp.bytes = in; sp.cand0 = 0; sp.enc_tab = bw->enc_tab; sp.R = m->R; sp.P = m->P; sp.cands = batch;
  stack_encode_dump_kernel<<<dim3(m->R, batch), kStkEpiThreads, 0, st>>>(sp, m->Cin, x0_out);
  dan_count_launch();
  DAN_CUDA_TRY(cudaGetLastError());
  return DAN_OK;
}

// FC input in the REFERENCE feature order (fp32), undoing the bf16 path's feature permutation (test hook)
namespace {
__global__ void fcin_to_reference_order_kernel(const uint4* __restrict__ fcin, long kstride, int rows, float* __restrict__ out,
                                               int fcIn, long permuted, long hw_base, int P, int C, int R, int bott) {
  const long total = (long)rows * fcIn;
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int k = (int)(i % fcIn); const long m = i / fcIn;
    out[m * fcIn + fc_ref_column(k, permuted, hw_base, P, C, R, bott)] =
        __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(fcin + m * kstride)[k]);      // kstride = pieces per row
  }
}
}  // namespace

int dan_bf16_debug_fc_input(dan_model* m, int batch, const void* ws, float* out, cudaStream_t st) {
  const Bf16Plan pl = make_plan(m, batch);
  const int nb = batch % pl.Bc == 0 ? pl.Bc : batch % pl.Bc;
  const uint4* FCIN = reinterpret_cast<const uint4*>(static_cast<const char*>(ws) + pl.off_fcin);
  const FcInLayout fl = fc_in_layout(m);
  fcin_to_reference_order_kernel<<<grid_for((long)nb * m->fcIn), 256, 0, st>>>(FCIN, pl.fcKC, nb, out, m->fcIn, fl.permuted, fl.hw_base, m->P, kC, m->R,
                                                                               m->bott > 0 ? m->bott : 1);
  DAN_CUDA_TRY(cudaGetLastError());
  return nb;
}
