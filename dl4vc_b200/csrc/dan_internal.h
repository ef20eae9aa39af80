// dan_internal.h — shared declarations of the DAN B200 library (not part of the public C-ABI).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stddef.h>
#include <mutex>
#include "../../include/dan_b200.h"

#define DAN_VOCAB 10
#define DAN_TILE_M 128           // rows (read positions) per GEMM tile, both precisions
#define DAN_HEAD_PAD 32          // the 27 head outputs are computed as one 32-wide GEMM

static inline int round_up_i(int x, int m) { return (x + m - 1) / m * m; }
static inline size_t round_up_z(size_t x, size_t m) { return (x + m - 1) / m * m; }

void dan_set_error(const char* fmt, ...);
// dan_inflate.cu: the launch behind dan_inflate_device, for callers that have checked their arguments (no argument checks)
int dan_inflate_launch(const uint8_t* src, const uint64_t* offsets, const uint32_t* lengths, int n, uint8_t* dst, uint64_t slot_bytes,
                       int32_t* status, cudaStream_t stream);
void dan_count_launch(int n = 1);
// kernel-class timing spans (no-ops unless dan_profile_enable(1)); classes: DAN_PROF_*
void dan_prof_begin(int cls, cudaStream_t st);
void dan_prof_end(int cls, cudaStream_t st);
struct DanProfScope {
  int cls; cudaStream_t st;
  DanProfScope(int c, cudaStream_t s) : cls(c), st(s) { dan_prof_begin(cls, st); }
  ~DanProfScope() { dan_prof_end(cls, st); }
};

#define DAN_CUDA_TRY(expr)                                                                      \
  do {                                                                                          \
    cudaError_t _e = (expr);                                                                    \
    if (_e != cudaSuccess) {                                                                    \
      dan_set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return DAN_E_CUDA;                                                                        \
    }                                                                                           \
  } while (0)

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) is per function AND per device: remember, per call site, the largest size already set
// on each device (a thread may move between devices, nn.DataParallel runs one thread per device) and raise it under a lock.
struct DanSmemAttr {
  std::mutex mu;
  size_t set_bytes[64] = {};
  template <class Kernel>
  cudaError_t ensure(Kernel kernel, size_t bytes) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    std::lock_guard<std::mutex> lk(mu);
    size_t& cur = set_bytes[dev & 63];
    if (bytes > cur) {
      e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
      if (e != cudaSuccess) return e;
      cur = bytes;
    }
    return cudaSuccess;
  }
};

// Row geometry of the activation matrices. Every per-read position is one row; reads are laid end to end with
// `gap` all-zero rows after each read (gap = largest dilation), so a dilated tap is a plain row offset and the
// zero padding of Conv2d(padding=(0,d)) (reference dl4vc/model.py:214-229) is implicit.
struct RowGeom {
  int P;          // positions per read (201)
  int R;          // reads per candidate (100)
  int gap;        // zero rows after each read
  int pitch;      // P + gap
  __host__ __device__ long rows_of(int cands) const { return (long)cands * R * pitch; }
};

struct DevInputs {
  const uint8_t* reads; const uint8_t* q; const uint8_t* strands;
  const uint8_t* ref; const uint8_t* ref_masks; const uint8_t* var_masks;
};

struct dan_model {
  dan_config cfg;
  int device;
  int L, C, Cin, CinPad, bott, P, R;
  RowGeom geom;
  int pooled, pooledPad;     // pooled feature count ((1|2)*C*P) and its 16-multiple
  int hwFeat;                // highway features entering the FC
  int fcIn, fcInPad;         // FC trunk input width
  int hidden;                // last FC width
  int pass_candidates;       // candidates per conv-stack pass
  int flags;                 // DAN_FLAG_* (dan_model_set_flags)
  bool loaded;
  // ---- fp32 packed weights (device). GEMM weights are stored K-major: W[k][n], n contiguous. ----
  float* emb; float* pe;
  float* convW[DAN_MAX_LAYERS];   // [3*CinPad or 3*C][C]   k = tap*Cin_pad + c
  float* convB[DAN_MAX_LAYERS];
  float* bnScale[DAN_MAX_LAYERS]; float* bnShift[DAN_MAX_LAYERS];   // eval BatchNorm folded: y*scale+shift
  float* resW[DAN_MAX_LAYERS];    // [C][C]
  float* resB[DAN_MAX_LAYERS];
  float* bottW[DAN_MAX_LAYERS];   // [C][bott]
  float* bottB[DAN_MAX_LAYERS];
  float* compW[DAN_MAX_LAYERS];   // [P*bott][bott]         k = p*bott + c
  float* compB[DAN_MAX_LAYERS];
  float* postW; float* postB;     // [pooledPad][D]
  float* fcW[DAN_MAX_FC];         // [KPad][N]
  float* fcB[DAN_MAX_FC];
  float* headW; float* headB;     // [hidden][32], [32]
  // ---- bf16 packed weights for the tcgen05 path (see dan_bf16.cu) ----
  void* bf16_store;               // opaque Bf16Weights*
  // ---- dan_forward_host: side stream + events for the double-buffered H2D staging ----
  cudaStream_t copy_stream; cudaEvent_t ev_copied[2], ev_done[2], ev_entry;
  std::mutex* host_mu;
};

// fp32 path (dan_fp32.cu)
size_t dan_fp32_workspace_bytes(const dan_model* m, int batch);
int dan_fp32_forward(dan_model* m, const DevInputs& in, int batch, float* heads_out, void* ws, size_t ws_bytes,
                     cudaStream_t st);
int dan_fp32_encode_reference_order(dan_model* m, const DevInputs& in, int batch, float* x0_out, cudaStream_t st);
int dan_fp32_debug_fc_input(dan_model* m, int batch, const void* ws, float* out, cudaStream_t st);
int dan_fp32_pack(dan_model* m, const dan_weights* w, cudaStream_t st);
void dan_fp32_free(dan_model* m);

// bf16 tcgen05 path (dan_bf16.cu)
// Candidates per FC-trunk chunk of the bf16 path: the whole number of conv-stack passes closest to 1024 candidates (PROD: 7 x 148 =
// 1036), so that a large batch is cut into full passes only (no ragged last pass per chunk). The 151 MB FC1 weight matrix is streamed once per chunk.
inline int dan_bf16_fc_chunk(const dan_model* m) {
  const int S = m->pass_candidates;
  if (S >= 1024) return S;
  const int n = (1024 + S / 2) / S;
  return (n < 1 ? 1 : n) * S;
}
size_t dan_bf16_workspace_bytes(const dan_model* m, int batch);
int dan_bf16_forward(dan_model* m, const DevInputs& in, int batch, float* heads_out, void* ws, size_t ws_bytes,
                     cudaStream_t st);
int dan_bf16_debug_fc_input(dan_model* m, int batch, const void* ws, float* out, cudaStream_t st);
int dan_bf16_encode_reference_order(dan_model* m, const DevInputs& in, int batch, float* x0_out, cudaStream_t st);
int dan_bf16_pack(dan_model* m, const dan_weights* w, cudaStream_t st);
void dan_bf16_free(dan_model* m);
int dan_bf16_supported(const dan_model* m);
const char* dan_bf16_unsupported_reason(const dan_model* m);     // nullptr when the bf16 path takes the configuration
int dan_bf16_route(const dan_model* m);                          // dan_model_bf16_route

// training path (dan_train.cu)
const char* dan_train_unsupported_reason(const dan_model* m);    // nullptr when the training kernels take the configuration
size_t dan_train_tape_bytes_impl(const dan_model* m, int batch);
int dan_train_forward_impl(dan_model* m, const dan_weights* w, const DevInputs& in, const uint8_t* removed, int batch, float dropout_p, uint64_t seed,
                           float* heads_out, void* tape, size_t tape_bytes, cudaStream_t st);
int dan_backward_impl(dan_model* m, const dan_weights* w, const DevInputs& in, const uint8_t* removed, int batch, float dropout_p, uint64_t seed,
                      const float* dheads, const float* heads_out, const dan_weights* grads, void* tape, size_t tape_bytes, cudaStream_t st);
