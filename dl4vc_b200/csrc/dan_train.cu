// dan_train.cu — training-mode forward and backward of the DAN (Basic2DNet with self.training: dl4vc/model.py:434-961,
// driven by dl4vc/trainer.py:213-217,426-439), fp32 on the CUDA-core FFMA kernels of the accuracy path.
//
// Forward differences from eval mode: BatchNorm normalises with the statistics of the batch (over batch x reads x positions,
// model.py:750-751) and updates the running statistics (momentum 0.1, unbiased variance); the three Dropout modules of the FC
// trunk (model.py:365-374) draw counter-based masks from (seed, element index); selected reads may be replaced by the empty-read
// encoding (model.py:633-716; the caller chooses which, like the reference's randperm). Every activation the backward pass needs
// is kept in a caller-provided tape.
//
// Backward: the same tap-gathering SGEMM with transposed weights and mirrored tap offsets for the data gradients, one
// "TN" SGEMM (reduction over rows, split over row ranges with a fixed-order finish) for every weight gradient, column sums for
// biases and the two BatchNorm reductions (double accumulation), element-wise masks, max / mean pool routing, the pool-add's
// read-axis broadcast, and a scatter-add into the 10 x 20 embedding table with nn.Embedding's scale_grad_by_freq.
#include <cstring>
#include "dan_fp32_kernels.cuh"

namespace {

constexpr int kRedRows = 1024;          // rows per partial of the column reductions
constexpr float kBnMomentum = 0.1f, kBnEps = 1e-5f;      // nn.BatchNorm2d defaults (model.py:217)

// ------------------------------------------------------------------------------------------------ column reductions
// part[chunk][which][c]: MODE 0: sum x | sum x^2 ; MODE 1: sum dy | sum dy * xhat, xhat = (u - mean) * rstd ; MODE 2: sum x
constexpr int kRedLanes = 8;             // row lanes per column: threads (c, lane) walk rows lane, lane + 8, ... of the partial's range
template <int MODE>
__global__ void __launch_bounds__(128 * kRedLanes) col_reduce_kernel(const float* __restrict__ X, int ldx, const float* __restrict__ U, int ldu,
                                                                     const double* __restrict__ mean, const double* __restrict__ rstd, long rows, int C,
                                                                     RowGeom g, int masked, double* __restrict__ part) {
  __shared__ double sh[2][kRedLanes][128];
  const int tx = threadIdx.x & 127, ry = threadIdx.x >> 7;
  const int c = blockIdx.y * 128 + tx;
  const long r0 = (long)blockIdx.x * kRedRows, r1 = r0 + kRedRows < rows ? r0 + kRedRows : rows;
  double s0 = 0.0, s1 = 0.0;
  if (c < C) {
    const double mu = MODE == 1 ? mean[c] : 0.0, rs = MODE == 1 ? rstd[c] : 0.0;
    int rp = masked ? (int)((r0 + ry) % g.pitch) : 0;                  // position of the row inside its read (rows >= P are gap rows)
#pragma unroll 4
    for (long r = r0 + ry; r < r1; r += kRedLanes) {
      const bool ok = !masked || rp < g.P;
      const float x = ok ? X[r * ldx + c] : 0.f;
      if (MODE == 0) { s0 += x; s1 += (double)x * x; }
      else if (MODE == 1) { const float u = ok ? U[r * ldu + c] : 0.f; s0 += x; s1 += (double)x * (((double)u - mu) * rs); }
      else s0 += x;
      if (masked) { rp += kRedLanes; if (rp >= g.pitch) rp -= g.pitch; }
    }
  }
  sh[0][ry][tx] = s0; sh[1][ry][tx] = s1;
  __syncthreads();
  if (ry == 0 && c < C) {              // lanes added in a fixed order
    double a0 = sh[0][0][tx], a1 = sh[1][0][tx];
#pragma unroll
    for (int k = 1; k < kRedLanes; ++k) { a0 += sh[0][k][tx]; a1 += sh[1][k][tx]; }
    part[((long)blockIdx.x * 2 + 0) * C + c] = a0;
    part[((long)blockIdx.x * 2 + 1) * C + c] = a1;
  }
}
// the partials of a column are added by 8 lanes (chunks k, k + 8, ...), lanes in a fixed order: one CTA of 128 x 8 threads per 128 columns
constexpr int kFinLanes = 8;
__device__ __forceinline__ void fin_sum(const double* __restrict__ part, int chunks, int C, int c, int lane, int tx, double (&sh)[2][kFinLanes][128], double& s0, double& s1) {
  double a0 = 0.0, a1 = 0.0;
  if (c < C)
    for (int k = lane; k < chunks; k += kFinLanes) { a0 += part[((long)k * 2 + 0) * C + c]; a1 += part[((long)k * 2 + 1) * C + c]; }
  sh[0][lane][tx] = a0; sh[1][lane][tx] = a1;
  __syncthreads();
  s0 = sh[0][0][tx]; s1 = sh[1][0][tx];
#pragma unroll
  for (int k = 1; k < kFinLanes; ++k) { s0 += sh[0][k][tx]; s1 += sh[1][k][tx]; }
}
__global__ void __launch_bounds__(128 * kFinLanes) bn_stats_finish_kernel(const double* __restrict__ part, int chunks, int C, double N, double* __restrict__ mean,
                                                                          double* __restrict__ rstd, float* __restrict__ run_mean, float* __restrict__ run_var) {
  __shared__ double sh[2][kFinLanes][128];
  const int tx = threadIdx.x & 127, lane = threadIdx.x >> 7, c = blockIdx.x * 128 + tx;
  double s0, s1;
  fin_sum(part, chunks, C, c, lane, tx, sh, s0, s1);
  if (lane != 0 || c >= C) return;
  const double m = s0 / N;
  double var = s1 / N - m * m;
  if (var < 0.0) var = 0.0;
  mean[c] = m;
  rstd[c] = 1.0 / sqrt(var + (double)kBnEps);
  if (run_mean) {      // running statistics: momentum 0.1, unbiased variance (torch.nn.functional.batch_norm)
    run_mean[c] = (1.f - kBnMomentum) * run_mean[c] + kBnMomentum * (float)m;
    run_var[c] = (1.f - kBnMomentum) * run_var[c] + kBnMomentum * (float)(var * N / (N - 1.0));
  }
}
// out0 / out1: sums of partial 0 / 1 (either may be null); out64_*: the same in double
__global__ void __launch_bounds__(128 * kFinLanes) col_finish_kernel(const double* __restrict__ part, int chunks, int C, float* __restrict__ out0, double* __restrict__ out64_0,
                                                                     float* __restrict__ out1, double* __restrict__ out64_1) {
  __shared__ double sh[2][kFinLanes][128];
  const int tx = threadIdx.x & 127, lane = threadIdx.x >> 7, c = blockIdx.x * 128 + tx;
  double s0, s1;
  fin_sum(part, chunks, C, c, lane, tx, sh, s0, s1);
  if (lane != 0 || c >= C) return;
  if (out0) out0[c] = (float)s0;
  if (out64_0) out64_0[c] = s0;
  if (out1) out1[c] = (float)s1;
  if (out64_1) out64_1[c] = s1;
}

// ------------------------------------------------------------------------------------------------ element-wise
__global__ void bn_apply_kernel(const float* __restrict__ U, float* __restrict__ Y, const double* __restrict__ mean, const double* __restrict__ rstd,
                                const float* __restrict__ gamma, const float* __restrict__ beta, long rows, int C, RowGeom g) {
  const long total = rows * C;
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const long r = i / C; const int c = (int)(i - r * C);
    Y[i] = (int)(r % g.pitch) < g.P ? (U[i] - (float)mean[c]) * (float)rstd[c] * gamma[c] + beta[c] : 0.f;
  }
}
// dZ = relu'(u) * dU, dU = gamma * rstd * (dY - dbeta / N - xhat * dgamma / N)   (BatchNorm after ReLU, model.py:749-751); no-BN: dZ = relu'(u) * dY
// The mean-removal is evaluated in double: sum(dY) and sum(dY * xhat) over 10^5-10^6 rows cancel against the per-row terms, and the conv bias /
// weight gradients downstream are sums over the rows that survive the ReLU mask — fp32 rounding of the two projections shows up there 1000-fold.
__global__ void bn_relu_bwd_kernel(const float* __restrict__ dY, const float* __restrict__ U, const double* __restrict__ mean, const double* __restrict__ rstd,
                                   const float* __restrict__ gamma, const double* __restrict__ dgamma, const double* __restrict__ dbeta, double invN,
                                   float* __restrict__ dZ, long rows, int C, RowGeom g, int use_bn) {
  const long total = rows * C;
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const long r = i / C; const int c = (int)(i - r * C);
    float v = 0.f;
    const float u = U[i];
    if ((int)(r % g.pitch) < g.P && u > 0.f) {
      if (use_bn) { const double xh = ((double)u - mean[c]) * rstd[c]; v = (float)((double)gamma[c] * rstd[c] * ((double)dY[i] - dbeta[c] * invN - xh * dgamma[c] * invN)); }
      else v = dY[i];
    }
    dZ[i] = v;
  }
}
__global__ void relu_mask_kernel(float* __restrict__ d, const float* __restrict__ act, long n) {      // d *= (act > 0)
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) if (!(act[i] > 0.f)) d[i] = 0.f;
}
__global__ void add_kernel(float* __restrict__ a, const float* __restrict__ b, long n) {
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) a[i] += b[i];
}
// counter-based dropout: keep element i of call `salt` iff hash(seed, salt, i) >= p * 2^32; kept values are scaled by 1 / (1 - p)
__device__ __forceinline__ uint32_t dropout_hash(uint64_t seed, uint32_t salt, uint64_t i) {
  uint64_t x = seed ^ (0x9E3779B97F4A7C15ull * (i + 1)) ^ ((uint64_t)salt << 56);
  x ^= x >> 30; x *= 0xBF58476D1CE4E5B9ull; x ^= x >> 27; x *= 0x94D049BB133111EBull; x ^= x >> 31;      // splitmix64 finaliser
  return (uint32_t)(x >> 32);
}
__global__ void dropout_kernel(const float* __restrict__ in, float* __restrict__ out, long n, float p, uint64_t seed, uint32_t salt) {
  const uint32_t thr = (uint32_t)fminf(p * 4294967296.f, 4294967295.f);
  const float scale = 1.f / (1.f - p);
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x)
    out[i] = (p > 0.f && dropout_hash(seed, salt, (uint64_t)i) < thr) ? 0.f : in[i] * (p > 0.f ? scale : 1.f);
}
// heads: d(loss)/d(pre-activation) from d(loss)/d(returned outputs): sigmoid on column 5, leaky_relu(0.01) on column 6 (model.py:954,956)
__global__ void head_act_bwd_kernel(const float* __restrict__ dout, const float* __restrict__ out, float* __restrict__ dz, int batch) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= batch * DAN_HEAD_PAD) return;
  const int b = i / DAN_HEAD_PAD, n = i - b * DAN_HEAD_PAD;
  float v = 0.f;
  if (n < DAN_NUM_HEAD_OUTPUTS) {
    v = dout[b * DAN_NUM_HEAD_OUTPUTS + n];
    const float o = out[b * DAN_NUM_HEAD_OUTPUTS + n];
    if (n == 5) v *= o * (1.f - o);
    else if (n == 6) v *= o >= 0.f ? 1.f : 0.01f;
  }
  dz[i] = v;
}

// ------------------------------------------------------------------------------------------------ pooling backward
// dH[cand, r, p, c] = dmean[cand, c, p] / R + (r == argmax_r H ? dmax[cand, c, p] : 0); dpooled in the reference feature order (max block | mean block,
// feature c * P + p, model.py:833-839); the arg-max is recomputed (first maximal row, like max_pool2d)
__global__ void pool_final_bwd_kernel(const float* __restrict__ H, int ldh, const float* __restrict__ dfc, int ld_dfc, float* __restrict__ dH, int C, RowGeom g, int skip_max) {
  const int cand = blockIdx.y, pp = blockIdx.x;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    const float* drow = dfc + (long)cand * ld_dfc;
    const float dmean = (skip_max ? drow[c * g.P + pp] : drow[(C + c) * g.P + pp]) / (float)g.R;
    int arg = -1; float mx = -INFINITY;
    if (!skip_max)
      for (int r = 0; r < g.R; ++r) { const float v = H[(((long)cand * g.R + r) * g.pitch + pp) * ldh + c]; if (v > mx) { mx = v; arg = r; } }
    const float dmax = skip_max ? 0.f : drow[c * g.P + pp];
    for (int r = 0; r < g.R; ++r) dH[(((long)cand * g.R + r) * g.pitch + pp) * ldh + c] = dmean + (r == arg ? dmax : 0.f);
  }
}
// d(hw[l][read][o]) from d(FC input): relu'(feature) * dfc at l*bott*R + o*R + r (concat) or relu'(mean over layers) * dfc / L (averaged)   (model.py:853-859)
__global__ void highway_bwd_kernel(const float* __restrict__ hw, long layer_stride, int L, int bott, int R, int concat, const float* __restrict__ fcin_feat,
                                   const float* __restrict__ dfc, int ld, float* __restrict__ dhw, int cands) {
  const int per = bott * R;
  const long total = (long)cands * L * per;
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int f = (int)(i % ((long)L * per)); const long cand = i / ((long)L * per);
    const int l = f / per, o = (f % per) / R, r = f % R;
    const int feat = concat ? f : f % per;
    const float act = fcin_feat[cand * ld + feat];
    const float d = act > 0.f ? dfc[cand * ld + feat] * (concat ? 1.f : 1.f / (float)L) : 0.f;
    dhw[l * layer_stride + (cand * R + r) * bott + o] = d;
  }
}

// ------------------------------------------------------------------------------------------------ "TN" SGEMM: weight gradients
// out[i][j] = sum over rows m of A[m][i] * B[m + b_off][j]   (i < I, j < J), rows split into `splits` ranges -> part[z][i][j]
struct TnParams {
  const float* A; int lda; const float* B; int ldb; long rows; int b_off; int I, J; float* part; int splits;
  float* out; long rs, cs; int Jkeep;      // splits == 1: written straight to out[i * rs + j * cs] (j < Jkeep)
};
__global__ void __launch_bounds__(256) sgemm_tn_kernel(TnParams p) {
  constexpr int BM = 128, BN = 128, BK = 16;
  __shared__ __align__(16) float As[2][BK][BM];
  __shared__ __align__(16) float Bs[2][BK][BN];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int i0 = blockIdx.x * BM, j0 = blockIdx.y * BN, z = blockIdx.z;
  const long per = ((p.rows + p.splits - 1) / p.splits + BK - 1) / BK * BK;
  const long m_begin = (long)z * per, m_end = m_begin + per < p.rows ? m_begin + per : p.rows;
  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
  float4 ra[2], rb[2];
  auto load = [&](long m0) {
#pragma unroll
    for (int v = 0; v < 2; ++v) {
      const int f = tid + v * 256, kk = f >> 5, cc = (f & 31) * 4;
      const long m = m0 + kk;
      const bool in = m < m_end;
      ra[v] = (in && i0 + cc < p.I) ? __ldg(reinterpret_cast<const float4*>(p.A + m * p.lda + i0 + cc)) : make_float4(0.f, 0.f, 0.f, 0.f);
      rb[v] = (in && j0 + cc < p.J) ? __ldg(reinterpret_cast<const float4*>(p.B + (m + p.b_off) * p.ldb + j0 + cc)) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  };
  auto store = [&](int buf) {
#pragma unroll
    for (int v = 0; v < 2; ++v) {
      const int f = tid + v * 256, kk = f >> 5, cc = (f & 31) * 4;
      *reinterpret_cast<float4*>(&As[buf][kk][cc]) = ra[v];
      *reinterpret_cast<float4*>(&Bs[buf][kk][cc]) = rb[v];
    }
  };
  if (m_begin < m_end) {
    load(m_begin);
    store(0);
    __syncthreads();
    int buf = 0;
    for (long m0 = m_begin; m0 < m_end; m0 += BK, buf ^= 1) {
      if (m0 + BK < m_end) load(m0 + BK);
#pragma unroll
      for (int k = 0; k < BK; ++k) {
        float a[8], b[8];
        *reinterpret_cast<float4*>(a) = *reinterpret_cast<const float4*>(&As[buf][k][ty * 4]);
        *reinterpret_cast<float4*>(a + 4) = *reinterpret_cast<const float4*>(&As[buf][k][64 + ty * 4]);
        *reinterpret_cast<float4*>(b) = *reinterpret_cast<const float4*>(&Bs[buf][k][tx * 4]);
        *reinterpret_cast<float4*>(b + 4) = *reinterpret_cast<const float4*>(&Bs[buf][k][64 + tx * 4]);
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
          for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
      }
      if (m0 + BK < m_end) { store(buf ^ 1); __syncthreads(); }
    }
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int ii = i0 + (i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4));
    if (ii >= p.I) continue;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int jj = j0 + (j < 4 ? tx * 4 + j : 64 + tx * 4 + (j - 4));
      if (p.splits == 1) { if (jj < p.Jkeep) p.out[ii * p.rs + jj * p.cs] = acc[i][j]; }
      else if (jj < p.J) p.part[((long)z * p.I + ii) * p.J + jj] = acc[i][j];
    }
  }
}
// out[i * rs + j * cs] = sum_z part[z][i][j] in split order (j < Jkeep)
__global__ void tn_finish_kernel(const float* __restrict__ part, int splits, int I, int J, int Jkeep, float* __restrict__ out, long rs, long cs) {
  const long total = (long)I * Jkeep;
  for (long t = blockIdx.x * (long)blockDim.x + threadIdx.x; t < total; t += (long)gridDim.x * blockDim.x) {
    const int i = (int)(t / Jkeep), j = (int)(t - (long)i * Jkeep);
    float v = 0.f;
    for (int z = 0; z < splits; ++z) v += part[((long)z * I + i) * J + j];
    out[i * rs + j * cs] = v;
  }
}
// compression weight gradient: temp [o][p * bott + c] -> torch layout (O, Cb, 1, P)
__global__ void comp_grad_permute_kernel(const float* __restrict__ tmp, float* __restrict__ out, int bott, int P) {
  const long total = (long)bott * bott * P;
  for (long t = blockIdx.x * (long)blockDim.x + threadIdx.x; t < total; t += (long)gridDim.x * blockDim.x) {
    const int pp = (int)(t % P); const long u = t / P; const int c = (int)(u % bott), o = (int)(u / bott);
    out[t] = tmp[(long)o * P * bott + (long)pp * bott + c];
  }
}

// ------------------------------------------------------------------------------------------------ weight layouts for the data gradients
// conv (Cout, Cin, 1, 3) -> [(tap, cout)][ld]: row k = tap * Cout + n holds w[n][c][tap] for c < Cin
__global__ void pack_conv_dgrad_kernel(const float* __restrict__ w, float* __restrict__ out, int Cout, int Cin, int ld) {
  const long total = (long)3 * Cout * ld;
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int c = (int)(i % ld); const long k = i / ld; const int n = (int)(k % Cout), t = (int)(k / Cout);
    out[i] = c < Cin ? w[((long)n * Cin + c) * 3 + t] : 0.f;
  }
}
// compression (O, Cb, 1, P) -> [o][p * Cb + c]
__global__ void pack_comp_dgrad_kernel(const float* __restrict__ w, float* __restrict__ out, int bott, int P) {
  const long total = (long)bott * P * bott;
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int c = (int)(i % bott); const long u = i / bott; const int pp = (int)(u % P), o = (int)(u / P);
    out[i] = w[((long)o * bott + c) * P + pp];
  }
}
// heads (27, hidden) -> (32, hidden), zero rows behind
__global__ void pad_rows_kernel(const float* __restrict__ w, float* __restrict__ out, int rows, int rows_pad, int cols) {
  const long total = (long)rows_pad * cols;
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) out[i] = i / cols < rows ? w[i] : 0.f;
}

// ------------------------------------------------------------------------------------------------ embedding backward
// dE[tok] = (sum of dX0 rows whose read token is tok, channels 0..D-1) / count_reads[tok] + (sum over reads of dX0 channels D..2D-1 at positions whose
// reference token is tok) / count_ref[tok]: two nn.Embedding calls with scale_grad_by_freq, padding_idx 0 (model.py:143-145,450-451). One block per
// candidate: partial table + counts per block, finished in block order.
__global__ void __launch_bounds__(240) emb_bwd_partial_kernel(const float* __restrict__ dX0, int ld, DevInputs in, const uint8_t* __restrict__ removed, int D, RowGeom g,
                                                              float* __restrict__ part /*[cand][2][10][D]*/, unsigned* __restrict__ cnt /*[cand][2][10]*/) {
  // thread = (channel c, group grp): private per-token sums over the group's share of the candidate's (position, read) cells, then a
  // fixed-order sum over the groups in shared memory (no floating-point atomics: bit-reproducible)
  extern __shared__ float sh[];                 // [groups][2][10][D]
  __shared__ unsigned cn[2 * DAN_VOCAB];
  const long cand = blockIdx.x;
  const int groups = blockDim.x / D, c = threadIdx.x % D, grp = threadIdx.x / D;
  const int P = g.P, R = g.R;
  if (threadIdx.x < 2 * DAN_VOCAB) cn[threadIdx.x] = 0u;
  __syncthreads();
  float accR[DAN_VOCAB], accF[DAN_VOCAB];
#pragma unroll
  for (int k = 0; k < DAN_VOCAB; ++k) { accR[k] = 0.f; accF[k] = 0.f; }
  if (grp < groups) {
    for (int idx = grp; idx < P * R; idx += groups) {
      const int pp = idx / R, r = idx - pp * R;
      const bool gone = removed && removed[cand * R + r];
      const unsigned tok = gone ? 0u : in.reads[(cand * P + pp) * R + r];
      const unsigned rtok = in.ref[cand * P + pp];
      const float* row = dX0 + (((long)cand * R + r) * g.pitch + pp) * ld;
      const float vr = row[c], vf = row[D + c];
#pragma unroll
      for (int k = 1; k < DAN_VOCAB; ++k) { accR[k] += tok == (unsigned)k ? vr : 0.f; accF[k] += rtok == (unsigned)k ? vf : 0.f; }
      if (c == 0) {
        if (tok < DAN_VOCAB) atomicAdd(&cn[tok], 1u);
        if (r == 0 && rtok < DAN_VOCAB) atomicAdd(&cn[DAN_VOCAB + rtok], 1u);
      }
    }
#pragma unroll
    for (int k = 0; k < DAN_VOCAB; ++k) { sh[((grp * 2 + 0) * DAN_VOCAB + k) * D + c] = accR[k]; sh[((grp * 2 + 1) * DAN_VOCAB + k) * D + c] = accF[k]; }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 2 * DAN_VOCAB * D; i += blockDim.x) {
    float v = 0.f;
    for (int gq = 0; gq < groups; ++gq) v += sh[gq * 2 * DAN_VOCAB * D + i];
    part[cand * 2 * DAN_VOCAB * D + i] = v;
  }
  for (int i = threadIdx.x; i < 2 * DAN_VOCAB; i += blockDim.x) cnt[cand * 2 * DAN_VOCAB + i] = cn[i];
}
__global__ void emb_bwd_finish_kernel(const float* __restrict__ part, const unsigned* __restrict__ cnt, int cands, int D, float* __restrict__ dE) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= DAN_VOCAB * D) return;
  const int tok = i / D;
  double s[2] = {0.0, 0.0};
  unsigned long long n[2] = {0, 0};
  for (int b = 0; b < cands; ++b)
    for (int w = 0; w < 2; ++w) { s[w] += part[((long)b * 2 + w) * DAN_VOCAB * D + i]; n[w] += cnt[((long)b * 2 + w) * DAN_VOCAB + tok]; }
  float v = 0.f;
  if (tok != 0) v = (float)((n[0] ? s[0] / (double)n[0] : 0.0) + (n[1] ? s[1] / (double)n[1] : 0.0));
  dE[i] = v;
}

// ------------------------------------------------------------------------------------------------ host side
inline int grid1d(long total, int block = 256) {
  long gsz = (total + block - 1) / block;
  return (int)(gsz < 1 ? 1 : (gsz > 148 * 16 ? 148 * 16 : gsz));
}

// row ranges of a weight-gradient product (sgemm_tn_kernel): enough of them for two CTAs per SM of a 148-SM part, at least 256 rows each
inline int tn_splits(long rows, int tiles) {
  long splits = (296 + tiles - 1) / tiles;
  if (splits > rows / 256) splits = rows / 256;
  return splits < 1 ? 1 : (int)splits;
}
constexpr int kLinearMaxSplits = 40;

struct TrainPlan {
  long rows, rowsAlloc, readsPad, hw_layer_stride;
  int BPad, chunks;
  size_t x0, u[DAN_MAX_LAYERS], y[DAN_MAX_LAYERS], h[DAN_MAX_LAYERS], inp[DAN_MAX_LAYERS], t[DAN_MAX_LAYERS], pool, hw, pooled, fcin, xd[DAN_MAX_FC + 1], act[DAN_MAX_FC],
      heads, stats, red, ga, gb, gt, dhw, dfc[2], dpooled, dz_heads, tnpart, wtmp, embpart, embcnt, total;
  size_t tn_part_floats;
};

TrainPlan make_train_plan(const dan_model* m, int B) {
  TrainPlan pl{};
  const RowGeom g = m->geom;
  const int C = m->C, L = m->L, bott = m->bott > 0 ? m->bott : 16;
  pl.rows = g.rows_of(B);
  pl.rowsAlloc = (pl.rows + 127) / 128 * 128 + 2L * g.gap + 128;
  pl.readsPad = ((long)B * m->R + 127) / 128 * 128;
  pl.hw_layer_stride = pl.readsPad * bott;
  pl.BPad = round_up_i(B, 128);
  pl.chunks = (int)((pl.rows + kRedRows - 1) / kRedRows);
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off += round_up_z(bytes, 256); return o; };
  const size_t rowC = (size_t)pl.rowsAlloc * C * 4;
  pl.x0 = take((size_t)pl.rowsAlloc * m->CinPad * 4);
  for (int l = 0; l < L; ++l) {
    pl.u[l] = take(l == 0 && m->CinPad > C ? (size_t)pl.rowsAlloc * m->CinPad * 4 : rowC);      // the backward writes d(x0) into U of layer 1
    pl.y[l] = m->cfg.use_batchnorm ? take(rowC) : pl.u[l];
    pl.h[l] = m->cfg.is_residual[l] ? take(rowC) : pl.y[l];
    pl.inp[l] = (l > 0 && m->cfg.pool_after[l - 1]) ? take(rowC) : 0;
    pl.t[l] = m->cfg.highway ? take(((size_t)pl.rowsAlloc + (size_t)128 * g.pitch) * bott * 4) : 0;
  }
  pl.pool = take((size_t)B * m->P * C * 4);
  pl.hw = take((size_t)L * pl.hw_layer_stride * 4);
  const size_t pooled_bytes = m->cfg.pool_combine_dimension > 0 ? (size_t)pl.BPad * m->pooledPad * 4 : 0;
  pl.pooled = take(pooled_bytes);                                  // input of the post-pool Linear (model.py:841-843); without it the pooled block heads FCIN
  pl.fcin = take((size_t)pl.BPad * m->fcInPad * 4);
  int K = m->fcInPad;
  for (int i = 0; i <= m->cfg.num_fc; ++i) {
    pl.xd[i] = take((size_t)pl.BPad * K * 4);                      // dropped-out input of FC layer i (i == num_fc: of the heads)
    if (i < m->cfg.num_fc) { K = m->cfg.fc_sizes[i]; pl.act[i] = take((size_t)pl.BPad * K * 4); }
  }
  pl.heads = take((size_t)pl.BPad * DAN_HEAD_PAD * 4);
  pl.stats = take((size_t)L * 4 * C * 8);                          // per layer (double): mean | rstd | dgamma | dbeta
  pl.red = take((size_t)pl.chunks * 2 * 1024 * 8 + 65536);
  // backward scratch
  pl.ga = take(rowC); pl.gb = take(rowC);
  pl.gt = m->cfg.highway ? take(((size_t)pl.rowsAlloc + (size_t)128 * g.pitch) * bott * 4) : 0;
  pl.dhw = take((size_t)L * pl.hw_layer_stride * 4);
  pl.dfc[0] = take((size_t)pl.BPad * m->fcInPad * 4); pl.dfc[1] = take((size_t)pl.BPad * m->fcInPad * 4);
  pl.dpooled = take(pooled_bytes);
  pl.dz_heads = take((size_t)pl.BPad * DAN_HEAD_PAD * 4);
  pl.tn_part_floats = (size_t)296 * 128 * 128 + (size_t)64 * bott * g.pitch * bott;      // conv-shaped problems | compression (I = bott, J = P*bott)
  const size_t fc_part = (size_t)kLinearMaxSplits * pl.BPad * 1024;                          // split-K partials of the small-M FC products (tr_linear)
  if (pl.tn_part_floats < fc_part) pl.tn_part_floats = fc_part;
  pl.tnpart = take(pl.tn_part_floats * 4);
  size_t wt = (size_t)3 * C * (C > m->CinPad ? C : m->CinPad);
  if ((size_t)bott * m->P * bott > wt) wt = (size_t)bott * m->P * bott;
  if ((size_t)DAN_HEAD_PAD * m->hidden > wt) wt = (size_t)DAN_HEAD_PAD * m->hidden;
  pl.wtmp = take(wt * 4);
  pl.embpart = take((size_t)B * 2 * DAN_VOCAB * m->cfg.embed_dim * 4);
  pl.embcnt = take((size_t)B * 2 * DAN_VOCAB * 4);
  pl.total = off;
  return pl;
}

int tr_gemm(const GemmParams& p, cudaStream_t st) { return launch_gemm(p, st); }

// A product with few output tiles and a long K (FC1: 32 x 73 856 -> 1024; the (1 x 201) compression: 3200 x 6432 -> 32) would run on a
// handful of CTAs: such products go split-K over fixed K ranges (partials in `part`, added in order by splitk_finish_kernel with the
// bias / ReLU), enough ranges for two CTAs per SM. Anything with a row mask, BatchNorm fold, residual or head activation runs unsplit.
int tr_gemm_auto(GemmParams q, float* part, size_t part_floats, cudaStream_t st) {
  const int bn = q.N <= 32 ? 32 : 128;
  const int tiles = ((q.M + 127) / 128) * ((q.N + bn - 1) / bn);
  const int K = q.ntaps * q.Kc;
  int splits = 1;
  if (part && !q.resid && !q.scale && !q.head_act && q.mask_pitch == 0 && tiles < 74 && K >= 4096) {
    splits = (296 + tiles - 1) / tiles;
    if (splits > kLinearMaxSplits) splits = kLinearMaxSplits;
    if (splits > K / 64) splits = K / 64;
    while (splits > 1 && (size_t)splits * q.M * q.N > part_floats) --splits;
  }
  if (splits <= 1) return launch_gemm(q, st);
  const float* bias = q.bias; const int relu = q.relu; float* out = q.out; const int ldo = q.ldo;
  q.out = part; q.ldo = q.N; q.splits = splits; q.split_stride = (long)q.M * q.N; q.bias = nullptr; q.relu = 0;
  int rc = launch_gemm(q, st);
  if (rc) return rc;
  splitk_finish_kernel<<<grid_for((long)q.M * q.N), 256, 0, st>>>(part, splits, q.split_stride, q.M, q.N, q.N, bias, relu, 0, out, ldo);
  dan_count_launch();
  DAN_CUDA_TRY(cudaGetLastError());
  return DAN_OK;
}

// y = [relu](x W + b) for a row-major activation matrix x [M][lda] and a K-major weight W[k][n]
int tr_linear(const float* A, int lda, int M, int K, const float* W, int N, int ldw, const float* bias, int relu, const float* resid, int ldr, float* out, int ldo,
              float* part, size_t part_floats, cudaStream_t st) {
  GemmParams q{};
  q.A = A; q.lda = lda; q.a_rows = M; q.M = M; q.ntaps = 1; q.tap_off[0] = 0; q.Kc = K;
  q.W = W; q.N = N; q.ldw = ldw; q.bias = bias; q.relu = relu; q.resid = resid; q.ldr = ldr; q.out = out; q.ldo = ldo; q.splits = 1;
  return tr_gemm_auto(q, part, part_floats, st);
}

// out[i * rs + j * cs] = sum_m A[m][i] * B[m + b_off][j]
int tr_wgrad(const float* A, int lda, const float* B, int ldb, long rows, int b_off, int I, int J, int Jkeep, float* out, long rs, long cs, float* part, size_t part_floats, cudaStream_t st) {
  int splits = tn_splits(rows, ((I + 127) / 128) * ((J + 127) / 128));
  while (splits > 1 && (size_t)splits * I * J > part_floats) --splits;
  TnParams p{A, lda, B, ldb, rows, b_off, I, J, part, splits, out, rs, cs, Jkeep};
  dim3 grid((unsigned)((I + 127) / 128), (unsigned)((J + 127) / 128), (unsigned)splits);
  sgemm_tn_kernel<<<grid, 256, 0, st>>>(p);
  if (splits > 1) tn_finish_kernel<<<grid1d((long)I * Jkeep), 256, 0, st>>>(part, splits, I, J, Jkeep, out, rs, cs);
  dan_count_launch(splits > 1 ? 2 : 1);
  DAN_CUDA_TRY(cudaGetLastError());
  return DAN_OK;
}

// out[c] = sum over rows of X[row][c]
int tr_colsum(const float* X, int ldx, long rows, int C, float* out, double* red, cudaStream_t st) {
  const int chunks = (int)((rows + kRedRows - 1) / kRedRows);
  RowGeom none{};
  col_reduce_kernel<2><<<dim3(chunks, (C + 127) / 128), 128 * kRedLanes, 0, st>>>(X, ldx, nullptr, 0, nullptr, nullptr, rows, C, none, 0, red);
  col_finish_kernel<<<(C + 127) / 128, 128 * kFinLanes, 0, st>>>(red, chunks, C, out, nullptr, nullptr, nullptr);
  dan_count_launch(2);
  DAN_CUDA_TRY(cudaGetLastError());
  return DAN_OK;
}

}  // namespace

size_t dan_train_tape_bytes_impl(const dan_model* m, int batch) { return make_train_plan(m, batch).total; }

const char* dan_train_unsupported_reason(const dan_model* m) {
  if (m->C % 4 || m->C > 1024) return "channels must be a multiple of 4, at most 1024";
  // the gradient of a residual layer fed by a pool-add (its residual bypasses the pool term, model.py:732 vs :742) is not implemented;
  // rejected here, before dan_train_forward has moved the BatchNorm running statistics
  for (int l = 1; l < m->L; ++l)
    if (m->cfg.pool_after[l - 1] && m->cfg.is_residual[l]) return "a residual layer directly behind a pool-add";
  return nullptr;
}

int dan_train_forward_impl(dan_model* m, const dan_weights* w, const DevInputs& in, const uint8_t* removed, int batch, float dropout_p, uint64_t seed,
                           float* heads_out, void* tape, size_t tape_bytes, cudaStream_t st) {
  const TrainPlan pl = make_train_plan(m, batch);
  if (tape_bytes < pl.total) { dan_set_error("training tape too small: %zu < %zu", tape_bytes, pl.total); return DAN_E_WORKSPACE; }
  char* base = static_cast<char*>(tape);
  const RowGeom g = m->geom;
  const int C = m->C, L = m->L, bott = m->bott, B = batch;
  const long lead = g.gap, rows = pl.rows;
  auto R_ = [&](size_t off, int ld) { return reinterpret_cast<float*>(base + off) + lead * ld; };
  int rc;
  // rows in front of / behind the data rows of every row matrix must read as zero (tap offsets reach them); the kernels below rewrite
  // all data rows themselves, gap rows between reads included (masked to zero)
  auto zero_edges = [&](size_t off, int ld) -> int {
    DAN_CUDA_TRY(cudaMemsetAsync(base + off, 0, (size_t)lead * ld * 4, st));
    DAN_CUDA_TRY(cudaMemsetAsync(base + off + ((size_t)lead + rows) * ld * 4, 0, (size_t)(pl.rowsAlloc - lead - rows) * ld * 4, st));
    return DAN_OK;
  };
  if ((rc = zero_edges(pl.x0, m->CinPad))) return rc;
  for (int l = 0; l < L; ++l) {
    if ((rc = zero_edges(pl.u[l], C))) return rc;
    if (pl.y[l] != pl.u[l] && (rc = zero_edges(pl.y[l], C))) return rc;
    if (pl.h[l] != pl.y[l] && (rc = zero_edges(pl.h[l], C))) return rc;
    if (pl.inp[l] && (rc = zero_edges(pl.inp[l], C))) return rc;
    if (m->cfg.highway) DAN_CUDA_TRY(cudaMemsetAsync(base + pl.t[l], 0, (size_t)lead * bott * 4, st));
  }
  float* X0 = R_(pl.x0, m->CinPad);
  {
    EncodeParams e{};
    e.in = in; e.emb = m->emb; e.pe = m->pe; e.D = m->cfg.embed_dim; e.Cin = m->Cin; e.CinPad = m->CinPad;
    e.use_q = m->cfg.use_q_scores; e.use_s = m->cfg.use_strands; e.use_m = m->cfg.use_reads_ref_var_mask; e.g = g; e.removed = removed;
    const size_t smem = encode_smem_bytes(m->P, m->R, m->cfg.embed_dim);
    static DanSmemAttr attr;
    DAN_CUDA_TRY(attr.ensure(encode_rows_fp32_kernel, smem));
    encode_rows_fp32_kernel<<<B, 256, smem, st>>>(e, 0, X0);
    dan_count_launch();
    DAN_CUDA_TRY(cudaGetLastError());
  }
  float* POOL = reinterpret_cast<float*>(base + pl.pool);
  float* HW = reinterpret_cast<float*>(base + pl.hw);
  double* STATS = reinterpret_cast<double*>(base + pl.stats);
  double* RED = reinterpret_cast<double*>(base + pl.red);
  const double N = (double)B * m->R * m->P;
  const float* cur = X0; int ld_cur = m->CinPad;
  for (int l = 0; l < L; ++l) {
    const int d = m->cfg.dilation[l];
    const float* conv_in = cur;
    if (l > 0 && m->cfg.pool_after[l - 1]) {
      float* hp = R_(pl.inp[l], C);
      add_pool_kernel<<<grid_for(rows * (C / 4)), 256, 0, st>>>(cur, POOL, hp, C, g, rows);
      dan_count_launch();
      conv_in = hp;
    }
    float* U = R_(pl.u[l], C);
    GemmParams p{};
    p.A = conv_in; p.lda = ld_cur; p.a_rows = pl.rowsAlloc - 2 * lead; p.M = (int)rows;
    p.ntaps = 3; p.tap_off[0] = -d; p.tap_off[1] = 0; p.tap_off[2] = d; p.Kc = (l == 0 ? m->CinPad : C);
    p.W = m->convW[l]; p.N = C; p.ldw = C; p.bias = m->convB[l]; p.relu = 1;
    p.mask_pitch = g.pitch; p.mask_valid = g.P; p.mask_total = rows; p.splits = 1; p.out = U; p.ldo = C;
    if ((rc = tr_gemm(p, st))) return rc;
    float* Y = R_(pl.y[l], C);
    if (m->cfg.use_batchnorm) {
      double* mean = STATS + (size_t)l * 4 * C; double* rstd = mean + C;
      col_reduce_kernel<0><<<dim3(pl.chunks, (C + 127) / 128), 128 * kRedLanes, 0, st>>>(U, C, nullptr, 0, nullptr, nullptr, rows, C, g, 1, RED);
      bn_stats_finish_kernel<<<(C + 127) / 128, 128 * kFinLanes, 0, st>>>(RED, pl.chunks, C, N, mean, rstd, const_cast<float*>(w->bn_mean[l]), const_cast<float*>(w->bn_var[l]));
      bn_apply_kernel<<<grid1d(rows * C), 256, 0, st>>>(U, Y, mean, rstd, w->bn_w[l], w->bn_b[l], rows, C, g);
      dan_count_launch(3);
    }
    float* H = R_(pl.h[l], C);
    if (m->cfg.is_residual[l]) {
      GemmParams q{};
      q.A = Y; q.lda = C; q.a_rows = pl.rowsAlloc - 2 * lead; q.M = (int)rows; q.ntaps = 1; q.tap_off[0] = 0; q.Kc = C;
      q.W = m->resW[l]; q.N = C; q.ldw = C; q.bias = m->resB[l];
      q.resid = cur; q.ldr = ld_cur;     // residual = layer input BEFORE the pool add (model.py:732)
      q.mask_pitch = g.pitch; q.mask_valid = g.P; q.mask_total = rows; q.out = H; q.ldo = C; q.splits = 1;
      if ((rc = tr_gemm(q, st))) return rc;
    }
    if (m->cfg.pool_after[l]) {
      pool_mean_kernel<<<dim3(g.P, B), 128, 0, st>>>(H, C, POOL, C, g);
      dan_count_launch();
    }
    if (m->cfg.highway) {
      float* T = reinterpret_cast<float*>(base + pl.t[l]) + lead * bott;
      GemmParams b{};
      b.A = H; b.lda = C; b.a_rows = pl.rowsAlloc - 2 * lead; b.M = (int)rows; b.ntaps = 1; b.tap_off[0] = 0; b.Kc = C;
      b.W = m->bottW[l]; b.N = bott; b.ldw = bott; b.bias = m->bottB[l]; b.relu = 1;
      b.mask_pitch = g.pitch; b.mask_valid = g.P; b.mask_total = rows; b.out = T; b.ldo = bott; b.splits = 1;
      if ((rc = tr_gemm(b, st))) return rc;
      GemmParams c{};   // (1x201) compression = one long dot product per read (model.py:776)
      c.A = T; c.lda = g.pitch * bott; c.a_rows = (long)B * m->R; c.M = B * m->R; c.ntaps = 1; c.tap_off[0] = 0;
      c.Kc = g.P * bott; c.W = m->compW[l]; c.N = bott; c.ldw = bott; c.bias = m->compB[l];
      c.out = HW + (long)l * pl.hw_layer_stride; c.ldo = bott; c.splits = 1;
      if ((rc = tr_gemm_auto(c, reinterpret_cast<float*>(base + pl.tnpart), pl.tn_part_floats, st))) return rc;
    }
    DAN_CUDA_TRY(cudaGetLastError());
    cur = H; ld_cur = C;
  }
  float* FCIN = reinterpret_cast<float*>(base + pl.fcin);
  DAN_CUDA_TRY(cudaMemsetAsync(FCIN, 0, (size_t)pl.BPad * m->fcInPad * 4, st));
  const int Dp = m->cfg.pool_combine_dimension;
  float* POOLED = Dp > 0 ? reinterpret_cast<float*>(base + pl.pooled) : FCIN;
  const int pooled_ld = Dp > 0 ? m->pooledPad : m->fcInPad;
  if (Dp > 0) DAN_CUDA_TRY(cudaMemsetAsync(POOLED, 0, (size_t)pl.BPad * m->pooledPad * 4, st));
  pool_final_kernel<<<dim3(g.P, B), 128, 0, st>>>(cur, C, POOLED, pooled_ld, C, g, m->cfg.skip_final_maxpool);
  dan_count_launch();
  if (Dp > 0) {      // post_pool_conv1D + ReLU (model.py:841-843) -> FC-input columns [0, D)
    if ((rc = tr_linear(POOLED, m->pooledPad, B, m->pooledPad, m->postW, Dp, Dp, m->postB, 1, nullptr, 0, FCIN, m->fcInPad,
                        reinterpret_cast<float*>(base + pl.tnpart), pl.tn_part_floats, st))) return rc;
  }
  if (m->cfg.highway) {
    highway_assemble_kernel<<<grid_for((long)B * m->hwFeat), 256, 0, st>>>(HW, pl.hw_layer_stride, L, bott, m->R, m->cfg.concat_hw_reads, FCIN + (Dp > 0 ? Dp : m->pooled),
                                                                          m->fcInPad, B);
    dan_count_launch();
  }
  // FC trunk: [Dropout] Linear ReLU Dropout ... (model.py:369-377), then the heads on the dropped-out last activation
  const float* x = FCIN; int K = m->fcInPad;
  for (int i = 0; i <= m->cfg.num_fc; ++i) {
    float* xd = reinterpret_cast<float*>(base + pl.xd[i]);
    dropout_kernel<<<grid1d((long)B * K), 256, 0, st>>>(x, xd, (long)B * K, dropout_p, seed, (uint32_t)i);
    dan_count_launch();
    if (i == m->cfg.num_fc) { x = xd; break; }
    float* a = reinterpret_cast<float*>(base + pl.act[i]);
    const int Nf = m->cfg.fc_sizes[i];
    if ((rc = tr_linear(xd, K, B, K, m->fcW[i], Nf, Nf, m->fcB[i], 1, nullptr, 0, a, Nf, reinterpret_cast<float*>(base + pl.tnpart), pl.tn_part_floats, st))) return rc;
    x = a; K = Nf;
  }
  float* HEADS = reinterpret_cast<float*>(base + pl.heads);
  {
    GemmParams q{};
    q.A = x; q.lda = K; q.a_rows = B; q.M = B; q.ntaps = 1; q.tap_off[0] = 0; q.Kc = K;
    q.W = m->headW; q.N = DAN_HEAD_PAD; q.ldw = DAN_HEAD_PAD; q.bias = m->headB; q.head_act = 1; q.out = HEADS; q.ldo = DAN_HEAD_PAD; q.splits = 1;
    if ((rc = tr_gemm(q, st))) return rc;
  }
  DAN_CUDA_TRY(cudaMemcpy2DAsync(heads_out, DAN_NUM_HEAD_OUTPUTS * 4, HEADS, DAN_HEAD_PAD * 4, DAN_NUM_HEAD_OUTPUTS * 4, B, cudaMemcpyDeviceToDevice, st));
  return DAN_OK;
}

int dan_backward_impl(dan_model* m, const dan_weights* w, const DevInputs& in, const uint8_t* removed, int batch, float dropout_p, uint64_t seed,
                      const float* dheads, const float* heads_out, const dan_weights* grads, void* tape, size_t tape_bytes, cudaStream_t st) {
  const TrainPlan pl = make_train_plan(m, batch);
  if (tape_bytes < pl.total) { dan_set_error("training tape too small: %zu < %zu", tape_bytes, pl.total); return DAN_E_WORKSPACE; }
  char* base = static_cast<char*>(tape);
  const RowGeom g = m->geom;
  const int C = m->C, L = m->L, bott = m->bott, B = batch, D = m->cfg.embed_dim;
  const long lead = g.gap, rows = pl.rows;
  auto R_ = [&](size_t off, int ld) { return reinterpret_cast<float*>(base + off) + lead * ld; };
  auto G_ = [](const float* p) { return const_cast<float*>(p); };      // gradient tensors are writable views of dan_weights
  int rc;
  double* STATS = reinterpret_cast<double*>(base + pl.stats);
  double* RED = reinterpret_cast<double*>(base + pl.red);
  float* TNP = reinterpret_cast<float*>(base + pl.tnpart);
  float* WT = reinterpret_cast<float*>(base + pl.wtmp);
  float* HW = reinterpret_cast<float*>(base + pl.hw);
  float* DHW = reinterpret_cast<float*>(base + pl.dhw);
  float* FCIN = reinterpret_cast<float*>(base + pl.fcin);
  const double invN = 1.0 / ((double)B * m->R * m->P);
  const float scale = dropout_p > 0.f ? 1.f / (1.f - dropout_p) : 1.f;
  (void)scale;

  // ---- heads ----
  float* DZ = reinterpret_cast<float*>(base + pl.dz_heads);
  head_act_bwd_kernel<<<(B * DAN_HEAD_PAD + 255) / 256, 256, 0, st>>>(dheads, heads_out, DZ, B);
  dan_count_launch();
  const int nfc = m->cfg.num_fc;
  const float* xd_heads = reinterpret_cast<const float*>(base + pl.xd[nfc]);
  if ((rc = tr_wgrad(DZ, DAN_HEAD_PAD, xd_heads, m->hidden, B, 0, DAN_HEAD_PAD, m->hidden, m->hidden, WT, m->hidden, 1, TNP, pl.tn_part_floats, st))) return rc;
  DAN_CUDA_TRY(cudaMemcpyAsync(G_(grads->head_w), WT, (size_t)DAN_NUM_HEAD_OUTPUTS * m->hidden * 4, cudaMemcpyDeviceToDevice, st));      // rows 27..31 are padding
  {
    float* hb = WT + (size_t)DAN_HEAD_PAD * m->hidden;      // wtmp holds at least 3*C*C floats
    if ((rc = tr_colsum(DZ, DAN_HEAD_PAD, B, DAN_HEAD_PAD, hb, RED, st))) return rc;
    DAN_CUDA_TRY(cudaMemcpyAsync(G_(grads->head_b), hb, DAN_NUM_HEAD_OUTPUTS * 4, cudaMemcpyDeviceToDevice, st));
  }
  float* dA = reinterpret_cast<float*>(base + pl.dfc[0]);
  float* dB = reinterpret_cast<float*>(base + pl.dfc[1]);
  pad_rows_kernel<<<grid1d((long)DAN_HEAD_PAD * m->hidden), 256, 0, st>>>(w->head_w, WT, DAN_NUM_HEAD_OUTPUTS, DAN_HEAD_PAD, m->hidden);
  dan_count_launch();
  // d(xd_heads) = dz . W_heads     (W' = torch (27 -> 32, hidden) read as [k = head output][n = hidden])
  if ((rc = tr_linear(DZ, DAN_HEAD_PAD, B, DAN_HEAD_PAD, WT, m->hidden, m->hidden, nullptr, 0, nullptr, 0, dA, m->hidden, TNP, pl.tn_part_floats, st))) return rc;
  // ---- FC trunk, last layer first ----
  int Nf = m->hidden;
  for (int i = nfc - 1; i >= 0; --i) {
    const int K = i == 0 ? m->fcInPad : m->cfg.fc_sizes[i - 1];
    const int Kreal = i == 0 ? m->fcIn : K;
    const float* act = reinterpret_cast<const float*>(base + pl.act[i]);
    const float* xd = reinterpret_cast<const float*>(base + pl.xd[i]);
    // dA holds d(dropped-out activation of layer i): undo dropout i+1 (same mask), then ReLU
    dropout_kernel<<<grid1d((long)B * Nf), 256, 0, st>>>(dA, dA, (long)B * Nf, dropout_p, seed, (uint32_t)(i + 1));
    relu_mask_kernel<<<grid1d((long)B * Nf), 256, 0, st>>>(dA, act, (long)B * Nf);
    dan_count_launch(2);
    if ((rc = tr_wgrad(dA, Nf, xd, K, B, 0, Nf, K, Kreal, G_(grads->fc_w[i]), Kreal, 1, TNP, pl.tn_part_floats, st))) return rc;
    if ((rc = tr_colsum(dA, Nf, B, Nf, G_(grads->fc_b[i]), RED, st))) return rc;
    // d(xd_i) = dpre . W_i: the torch weight (N, K) row-major is the K-major operand of this product; layer 0 has K = fcIn columns (ld fcIn) against fcInPad rows of xd
    if ((rc = tr_linear(dA, Nf, B, Nf, w->fc_w[i], Kreal, Kreal, nullptr, 0, nullptr, 0, dB, K, TNP, pl.tn_part_floats, st))) return rc;
    { float* t = dA; dA = dB; dB = t; }
    Nf = K;
  }
  // dA = d(dropped-out FC input) [B][fcInPad]: undo dropout 0
  dropout_kernel<<<grid1d((long)B * m->fcInPad), 256, 0, st>>>(dA, dA, (long)B * m->fcInPad, dropout_p, seed, 0u);
  dan_count_launch();
  // ---- post-pool Linear: dA[:, 0:D) through its ReLU, weight / bias gradients, data gradient into the pooled features ----
  const int Dp = m->cfg.pool_combine_dimension;
  const float* dpooled = dA;
  int dpooled_ld = m->fcInPad;
  if (Dp > 0) {
    relu_mask_kernel<<<grid1d((long)B * m->fcInPad), 256, 0, st>>>(dA, FCIN, (long)B * m->fcInPad);      // the highway block is masked alike below
    dan_count_launch();
    const float* POOLED = reinterpret_cast<const float*>(base + pl.pooled);
    if ((rc = tr_wgrad(dA, m->fcInPad, POOLED, m->pooledPad, B, 0, Dp, m->pooledPad, m->pooled, G_(grads->post_pool_w), m->pooled, 1, TNP, pl.tn_part_floats, st))) return rc;
    if ((rc = tr_colsum(dA, m->fcInPad, B, Dp, G_(grads->post_pool_b), RED, st))) return rc;
    float* DP = reinterpret_cast<float*>(base + pl.dpooled);
    // d(pooled) = dpre . W_post: the torch weight (D, pooled) row-major is the K-major operand of this product
    if ((rc = tr_linear(dA, m->fcInPad, B, Dp, w->post_pool_w, m->pooled, m->pooled, nullptr, 0, nullptr, 0, DP, m->pooledPad, TNP, pl.tn_part_floats, st))) return rc;
    dpooled = DP; dpooled_ld = m->pooledPad;
  }
  // ---- highway features and final pools ----
  if (m->cfg.highway) {
    const int hw0 = Dp > 0 ? Dp : m->pooled;
    highway_bwd_kernel<<<grid1d((long)B * L * bott * m->R), 256, 0, st>>>(HW, pl.hw_layer_stride, L, bott, m->R, m->cfg.concat_hw_reads, FCIN + hw0, dA + hw0,
                                                                         m->fcInPad, DHW, B);
    dan_count_launch();
  }
  float* GA = R_(pl.ga, C);      // d(layer output) of the layer being processed
  float* GB = R_(pl.gb, C);
  DAN_CUDA_TRY(cudaMemsetAsync(base + pl.ga, 0, pl.dhw - pl.ga, st));      // gap rows of the gradient row matrices
  pool_final_bwd_kernel<<<dim3(g.P, B), 128, 0, st>>>(R_(pl.h[L - 1], C), C, dpooled, dpooled_ld, GA, C, g, m->cfg.skip_final_maxpool);
  dan_count_launch();
  DAN_CUDA_TRY(cudaGetLastError());
  float* POOLG = reinterpret_cast<float*>(base + pl.pool);      // forward's pool table is dead by now: reused for the pool-add backward
  for (int l = L - 1; l >= 0; --l) {
    const int d = m->cfg.dilation[l];
    const int cin = l == 0 ? m->Cin : C, cinPad = l == 0 ? m->CinPad : C;
    const float* H = R_(pl.h[l], C);
    const float* Y = R_(pl.y[l], C);
    const float* U = R_(pl.u[l], C);
    const float* IN = l == 0 ? R_(pl.x0, m->CinPad) : R_(pl.h[l - 1], C);                  // layer input without the pool term
    const float* CONV_IN = (l > 0 && m->cfg.pool_after[l - 1]) ? R_(pl.inp[l], C) : IN;
    // ---- highway branch of this layer: compression (1 x P) conv and bottleneck 1x1 ----
    if (m->cfg.highway) {
      float* T = reinterpret_cast<float*>(base + pl.t[l]) + lead * bott;
      float* GT = reinterpret_cast<float*>(base + pl.gt) + lead * bott;
      const float* dhw = DHW + (long)l * pl.hw_layer_stride;
      const int reads = B * m->R, KT = g.P * bott;
      // dWc[o][(p, c)] = sum_reads dhw[read][o] * T[read][(p, c)] -> torch (O, Cb, 1, P)
      if ((rc = tr_wgrad(dhw, bott, T, g.pitch * bott, reads, 0, bott, KT, KT, WT, KT, 1, TNP, pl.tn_part_floats, st))) return rc;
      comp_grad_permute_kernel<<<grid1d((long)bott * KT), 256, 0, st>>>(WT, G_(grads->comp_w[l]), bott, g.P);
      dan_count_launch();
      if ((rc = tr_colsum(dhw, bott, reads, bott, G_(grads->comp_b[l]), RED, st))) return rc;
      // dT[read][(p, c)] = dhw[read][:] . Wc[:][c][p]
      pack_comp_dgrad_kernel<<<grid1d((long)bott * KT), 256, 0, st>>>(w->comp_w[l], WT, bott, g.P);
      dan_count_launch();
      {
        GemmParams q{};
        q.A = dhw; q.lda = bott; q.a_rows = reads; q.M = reads; q.ntaps = 1; q.tap_off[0] = 0; q.Kc = bott;
        q.W = WT; q.N = KT; q.ldw = KT; q.out = GT; q.ldo = g.pitch * bott; q.splits = 1;
        if ((rc = tr_gemm(q, st))) return rc;
      }
      relu_mask_kernel<<<grid1d(rows * bott), 256, 0, st>>>(GT, T, rows * bott);
      dan_count_launch();
      if ((rc = tr_wgrad(GT, bott, H, C, rows, 0, bott, C, C, G_(grads->bott_w[l]), C, 1, TNP, pl.tn_part_floats, st))) return rc;
      if ((rc = tr_colsum(GT, bott, rows, bott, G_(grads->bott_b[l]), RED, st))) return rc;
      // dH += dT . Wb      (torch (bott, C) read as [k = bottleneck channel][n = C])
      {
        GemmParams q{};
        q.A = GT; q.lda = bott; q.a_rows = pl.rowsAlloc - 2 * lead; q.M = (int)rows; q.ntaps = 1; q.tap_off[0] = 0; q.Kc = bott;
        q.W = w->bott_w[l]; q.N = C; q.ldw = C; q.resid = GA; q.ldr = C; q.out = GA; q.ldo = C; q.splits = 1;
        if ((rc = tr_gemm(q, st))) return rc;
      }
    }
    // ---- residual 1x1: h = Wres y + b + in ----
    const float* dY = GA;
    if (m->cfg.is_residual[l]) {
      if ((rc = tr_wgrad(GA, C, Y, C, rows, 0, C, C, C, G_(grads->res_w[l]), C, 1, TNP, pl.tn_part_floats, st))) return rc;
      if ((rc = tr_colsum(GA, C, rows, C, G_(grads->res_b[l]), RED, st))) return rc;
      GemmParams q{};
      q.A = GA; q.lda = C; q.a_rows = pl.rowsAlloc - 2 * lead; q.M = (int)rows; q.ntaps = 1; q.tap_off[0] = 0; q.Kc = C;
      q.W = w->res_w[l]; q.N = C; q.ldw = C; q.out = GB; q.ldo = C; q.splits = 1;
      q.mask_pitch = g.pitch; q.mask_valid = g.P; q.mask_total = rows;
      if ((rc = tr_gemm(q, st))) return rc;
      dY = GB;
    }
    // ---- BatchNorm (batch statistics) and ReLU ----
    double* mean = STATS + (size_t)l * 4 * C; double* rstd = mean + C; double* dgamma = mean + 2 * C; double* dbeta = mean + 3 * C;
    float* DZl = const_cast<float*>(dY) == GA ? GB : GB;      // dZ always lands in GB (element-wise, in place when dY == GB)
    if (m->cfg.use_batchnorm) {
      col_reduce_kernel<1><<<dim3(pl.chunks, (C + 127) / 128), 128 * kRedLanes, 0, st>>>(dY, C, U, C, mean, rstd, rows, C, g, 1, RED);
      col_finish_kernel<<<(C + 127) / 128, 128 * kFinLanes, 0, st>>>(RED, pl.chunks, C, G_(grads->bn_b[l]), dbeta, G_(grads->bn_w[l]), dgamma);
      dan_count_launch(2);
    }
    bn_relu_bwd_kernel<<<grid1d(rows * C), 256, 0, st>>>(dY, U, mean, rstd, w->bn_w[l], dgamma, dbeta, invN, DZl, rows, C, g, m->cfg.use_batchnorm);
    dan_count_launch();
    // ---- conv (1x3, dilation d): weight / bias gradients, then the data gradient ----
    if ((rc = tr_colsum(DZl, C, rows, C, G_(grads->conv_b[l]), RED, st))) return rc;
    for (int t = 0; t < 3; ++t) {
      // dW[cout][cin][tap] = sum_m dZ[m][cout] * conv_in[m + (t-1) d][cin]
      if ((rc = tr_wgrad(DZl, C, CONV_IN, cinPad, rows, (t - 1) * d, C, cinPad, cin, G_(grads->conv_w[l]) + t, (long)cin * 3, 3, TNP, pl.tn_part_floats, st))) return rc;
    }
    if (l == 0 && !grads->embeddings) break;
    pack_conv_dgrad_kernel<<<grid1d((long)3 * C * cinPad), 256, 0, st>>>(w->conv_w[l], WT, C, cin, cinPad);
    dan_count_launch();
    {
      // d(conv_in)[m][cin] = sum_tap dZ[m - (t-1) d][:] . w[:, cin, tap]: the same tap-gathering GEMM with mirrored offsets
      float* DIN = (l == 0) ? R_(pl.u[0], m->CinPad) : GA;      // layer 1: its (dead) U matrix takes d(x0) (sized for max(C, CinPad) columns)
      GemmParams q{};
      q.A = DZl; q.lda = C; q.a_rows = pl.rowsAlloc - 2 * lead; q.M = (int)rows;
      q.ntaps = 3; q.tap_off[0] = d; q.tap_off[1] = 0; q.tap_off[2] = -d; q.Kc = C;
      q.W = WT; q.N = cinPad; q.ldw = cinPad; q.out = DIN; q.ldo = l == 0 ? m->CinPad : C; q.splits = 1;
      q.mask_pitch = g.pitch; q.mask_valid = g.P; q.mask_total = rows;
      if (l > 0 && m->cfg.is_residual[l] && !(m->cfg.pool_after[l - 1])) { /* residual pass-through is added below */ }
      // the residual pass-through d(in) += d(h) needs GA intact until the GEMM has read ... GA is only the OUTPUT here (A = DZl in GB): safe to overwrite after saving the pass-through
      if (l > 0 && m->cfg.is_residual[l]) {
        // DIN = conv dgrad + dH (pass-through): sgemm adds resid[m][n] element-wise, in place on GA
        q.resid = GA; q.ldr = C;
      }
      if ((rc = tr_gemm(q, st))) return rc;
      if (l == 0) {
        // ---- embedding table ----
        float* part = reinterpret_cast<float*>(base + pl.embpart);
        unsigned* cnt = reinterpret_cast<unsigned*>(base + pl.embcnt);
        const int groups = 240 / D;
        const size_t sh = (size_t)groups * 2 * DAN_VOCAB * D * 4;
        emb_bwd_partial_kernel<<<B, groups * D, sh, st>>>(DIN, m->CinPad, in, removed, D, g, part, cnt);
        emb_bwd_finish_kernel<<<(DAN_VOCAB * D + 127) / 128, 128, 0, st>>>(part, cnt, B, D, G_(grads->embeddings));
        dan_count_launch(2);
        break;
      }
    }
    // ---- pool-add in front of this layer: in = h + mean_r(h)  =>  dh = din + mean_r(din); with a residual the pass-through bypasses the pool term ----
    if (m->cfg.pool_after[l - 1]) {
      if (m->cfg.is_residual[l]) { dan_set_error("training: a residual layer directly behind a pool-add is not supported"); return DAN_E_UNSUPPORTED; }
      pool_mean_kernel<<<dim3(g.P, B), 128, 0, st>>>(GA, C, POOLG, C, g);
      add_pool_kernel<<<grid_for(rows * (C / 4)), 256, 0, st>>>(GA, POOLG, GA, C, g, rows);
      dan_count_launch(2);
    }
    DAN_CUDA_TRY(cudaGetLastError());
  }
  DAN_CUDA_TRY(cudaGetLastError());
  return DAN_OK;
}
