// dan_capi.cu — the extern "C" boundary declared in include/dan_b200.h.
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <new>
#include "dan_internal.h"
#include "dan_records.h"

#include <vector>
#include <mutex>

namespace {
thread_local char g_error[512] = "";
thread_local int g_launches = 0;

// ---- optional per-kernel-class timing (CUDA events on the launching stream; off by default) ----
struct ProfSpan { cudaEvent_t a, b; int cls; };
std::mutex g_prof_mu;
bool g_prof_on = false;
std::vector<ProfSpan> g_prof_spans;
std::vector<cudaEvent_t> g_prof_pool;
cudaEvent_t prof_event() {
  if (!g_prof_pool.empty()) { cudaEvent_t e = g_prof_pool.back(); g_prof_pool.pop_back(); return e; }
  cudaEvent_t e = nullptr;
  cudaEventCreate(&e);
  return e;
}
}  // namespace

void dan_prof_begin(int cls, cudaStream_t st) {
  if (!g_prof_on) return;
  std::lock_guard<std::mutex> lk(g_prof_mu);
  ProfSpan s{prof_event(), prof_event(), cls};
  cudaEventRecord(s.a, st);
  g_prof_spans.push_back(s);
}
void dan_prof_end(int cls, cudaStream_t st) {
  if (!g_prof_on) return;
  std::lock_guard<std::mutex> lk(g_prof_mu);
  for (size_t i = g_prof_spans.size(); i-- > 0;)
    if (g_prof_spans[i].cls == cls) { cudaEventRecord(g_prof_spans[i].b, st); break; }
}

void dan_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_error, sizeof(g_error), fmt, ap);
  va_end(ap);
}
void dan_count_launch(int n) { g_launches += n; }

// scores[b] = {1 - softmax(xbinary)[0], softmax(xVT)[0..2]}  (trainer.py:611-623); one thread per candidate
__global__ void dan_scores_kernel(const float* __restrict__ heads, int batch, float4* __restrict__ scores) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= batch) return;
  const float* h = heads + (long)b * DAN_NUM_HEAD_OUTPUTS;
  const float b0 = h[0], b1 = h[1], v0 = h[2], v1 = h[3], v2 = h[4];
  const float mb = fmaxf(b0, b1), e0 = expf(b0 - mb), e1 = expf(b1 - mb);
  const float mv = fmaxf(v0, fmaxf(v1, v2)), f0 = expf(v0 - mv), f1 = expf(v1 - mv), f2 = expf(v2 - mv), inv = 1.f / (f0 + f1 + f2);
  scores[b] = make_float4(1.f - e0 / (e0 + e1), f0 * inv, f1 * inv, f2 * inv);
}


extern "C" {

const char* dan_last_error(void) { return g_error; }
const char* dan_version(void) { return "dan_b200 0.1 sm_100a"; }
int dan_last_launch_count(void) { return g_launches; }

int dan_profile_enable(int on) {
  std::lock_guard<std::mutex> lk(g_prof_mu);
  g_prof_on = on != 0;
  for (auto& s : g_prof_spans) { g_prof_pool.push_back(s.a); g_prof_pool.push_back(s.b); }
  g_prof_spans.clear();
  return DAN_OK;
}

int dan_profile_read(double* ms_by_class, int* launches_by_class, int num_classes) {
  if (!ms_by_class || !launches_by_class || num_classes < 1) { dan_set_error("bad argument"); return DAN_E_INVALID; }
  std::lock_guard<std::mutex> lk(g_prof_mu);
  for (int i = 0; i < num_classes; ++i) { ms_by_class[i] = 0.0; launches_by_class[i] = 0; }
  for (auto& s : g_prof_spans) {
    if (cudaEventSynchronize(s.b) != cudaSuccess) { dan_set_error("profile event not recorded"); return DAN_E_CUDA; }
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, s.a, s.b) != cudaSuccess) { dan_set_error("cudaEventElapsedTime failed"); return DAN_E_CUDA; }
    if (s.cls >= 0 && s.cls < num_classes) { ms_by_class[s.cls] += ms; launches_by_class[s.cls] += 1; }
  }
  return (int)g_prof_spans.size();
}

const char* dan_profile_class_name(int cls) {
  static const char* names[DAN_PROF_NUM_CLASSES] = {"conv_stack", "gemm", "encode", "pool_elementwise"};
  return (cls >= 0 && cls < DAN_PROF_NUM_CLASSES) ? names[cls] : "";
}

int dan_model_create(const dan_config* cfg, dan_model** out) {
  if (!cfg || !out) { dan_set_error("null argument"); return DAN_E_INVALID; }
  *out = nullptr;
  const dan_config& c = *cfg;
  if (c.total_conv_layers < 1 || c.total_conv_layers > DAN_MAX_LAYERS) { dan_set_error("total_conv_layers %d out of range 1..%d", c.total_conv_layers, DAN_MAX_LAYERS); return DAN_E_UNSUPPORTED; }
  if (c.channels < 16 || c.channels % 16) { dan_set_error("channels must be a multiple of 16 (got %d)", c.channels); return DAN_E_UNSUPPORTED; }
  if (c.embed_dim < 1 || c.embed_dim > 64) { dan_set_error("embed_dim %d unsupported", c.embed_dim); return DAN_E_UNSUPPORTED; }
  if (c.num_fc < 1 || c.num_fc > DAN_MAX_FC) { dan_set_error("layer_sizes must have 1..%d entries", DAN_MAX_FC); return DAN_E_UNSUPPORTED; }
  for (int i = 0; i < c.num_fc; ++i)
    if (c.fc_sizes[i] < 16 || c.fc_sizes[i] % 16) { dan_set_error("FC width %d must be a multiple of 16", c.fc_sizes[i]); return DAN_E_UNSUPPORTED; }
  if (c.highway && (c.bottleneck < 16 || c.bottleneck % 16 || c.bottleneck > 64)) { dan_set_error("bottleneck size must be 16, 32, 48 or 64 (got %d)", c.bottleneck); return DAN_E_UNSUPPORTED; }
  if (c.num_reads < 1 || c.read_len < 3) { dan_set_error("bad pileup shape %d x %d", c.num_reads, c.read_len); return DAN_E_INVALID; }
  if (c.pool_combine_dimension < 0 || (c.pool_combine_dimension % 16)) { dan_set_error("pool_combine_dimension must be a multiple of 16"); return DAN_E_UNSUPPORTED; }
  int gap = 1;
  for (int l = 0; l < c.total_conv_layers; ++l) {
    if (c.dilation[l] < 1 || c.dilation[l] > 8) { dan_set_error("dilation %d of layer %d unsupported (1..8)", c.dilation[l], l + 1); return DAN_E_UNSUPPORTED; }
    if (c.dilation[l] > gap) gap = c.dilation[l];
    if (c.is_residual[l] && l == 0) { dan_set_error("layer 1 cannot be residual (channel mismatch; model.py:28,209)"); return DAN_E_UNSUPPORTED; }
  }
  if (c.pool_after[c.total_conv_layers - 1]) { /* harmless: pooled after the last layer is never consumed */ }
  dan_model* m = new (std::nothrow) dan_model();
  if (!m) { dan_set_error("out of host memory"); return DAN_E_INVALID; }
  memset(m, 0, sizeof(*m));
  m->cfg = c;
  if (cudaGetDevice(&m->device) != cudaSuccess) { delete m; dan_set_error("no CUDA device"); return DAN_E_CUDA; }
  m->L = c.total_conv_layers; m->C = c.channels; m->bott = c.highway ? c.bottleneck : 0;
  m->P = c.read_len; m->R = c.num_reads;
  m->Cin = 2 * c.embed_dim + (c.use_q_scores ? 1 : 0) + (c.use_strands ? 1 : 0) + (c.use_reads_ref_var_mask ? 3 : 0);
  m->CinPad = round_up_i(m->Cin, 16);
  m->geom.P = m->P; m->geom.R = m->R; m->geom.gap = gap; m->geom.pitch = m->P + gap;
  m->pooled = (c.skip_final_maxpool ? 1 : 2) * m->C * m->P;
  m->pooledPad = round_up_i(m->pooled, 16);
  m->hwFeat = c.highway ? (c.concat_hw_reads ? m->L : 1) * m->bott * m->R : 0;
  m->fcIn = (c.pool_combine_dimension > 0 ? c.pool_combine_dimension : m->pooled) + m->hwFeat;
  m->fcInPad = round_up_i(m->fcIn, 16);
  m->hidden = c.fc_sizes[c.num_fc - 1];
  int sms = 148;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, m->device);
  m->pass_candidates = sms;    // one candidate per CTA of the persistent stack kernel (B200: 148 candidates x 100 reads = 100 reads per CTA, no tail imbalance)
  m->host_mu = new std::mutex();
  *out = m;
  return DAN_OK;
}

int dan_model_destroy(dan_model* m) {
  if (!m) return DAN_OK;
  dan_fp32_free(m);
  dan_bf16_free(m);
  if (m->copy_stream) {
    cudaStreamDestroy(m->copy_stream);
    for (int i = 0; i < 2; ++i) { cudaEventDestroy(m->ev_copied[i]); cudaEventDestroy(m->ev_done[i]); }
    cudaEventDestroy(m->ev_entry);
  }
  delete m->host_mu;
  delete m;
  return DAN_OK;
}

int dan_model_load_weights(dan_model* m, const dan_weights* w, void* stream) {
  if (!m || !w) { dan_set_error("null argument"); return DAN_E_INVALID; }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int rc = dan_fp32_pack(m, w, st);
  if (rc) return rc;
  if (dan_bf16_supported(m)) {
    rc = dan_bf16_pack(m, w, st);
    if (rc) return rc;
  }
  m->loaded = true;
  return DAN_OK;
}

int dan_model_set_pass_candidates(dan_model* m, int candidates) {
  if (!m || candidates < 1) { dan_set_error("pass_candidates must be >= 1"); return DAN_E_INVALID; }
  m->pass_candidates = candidates;
  return DAN_OK;
}

int dan_model_set_flags(dan_model* m, int flags) {
  if (!m || (flags & ~DAN_FLAG_LAYERWISE)) { dan_set_error("unknown flag bits %d", flags); return DAN_E_INVALID; }
  m->flags = flags;
  return DAN_OK;
}

int dan_model_bf16_route(const dan_model* m) {
  if (!m) { dan_set_error("null model"); return DAN_E_INVALID; }
  return dan_bf16_route(m);
}

size_t dan_workspace_bytes(const dan_model* m, int batch, int precision) {
  if (!m || batch < 0) return 0;
  if (precision == DAN_PRECISION_BF16) return dan_bf16_workspace_bytes(m, batch);
  return dan_fp32_workspace_bytes(m, batch);
}

static int check_forward_args(dan_model* m, int precision, const uint8_t* reads, const uint8_t* q, const uint8_t* s,
                              const uint8_t* ref, const uint8_t* rm, const uint8_t* vm, int batch, const void* out) {
  if (!m) { dan_set_error("null model"); return DAN_E_INVALID; }
  if (!m->loaded) { dan_set_error("dan_model_load_weights has not been called"); return DAN_E_INVALID; }
  if (batch < 0) { dan_set_error("negative batch"); return DAN_E_INVALID; }
  if (batch > 0 && (!reads || !ref || !out)) { dan_set_error("reads / ref / output pointer is null"); return DAN_E_INVALID; }
  if (batch > 0 && m->cfg.use_q_scores && !q) { dan_set_error("model uses q-scores but q_scores is null (model.py:534)"); return DAN_E_INVALID; }
  if (batch > 0 && m->cfg.use_strands && !s) { dan_set_error("model uses strands but strands is null (model.py:549)"); return DAN_E_INVALID; }
  if (batch > 0 && m->cfg.use_reads_ref_var_mask && (!rm || !vm)) { dan_set_error("model uses ref/var masks but a mask pointer is null (model.py:576)"); return DAN_E_INVALID; }
  if (precision != DAN_PRECISION_FP32 && precision != DAN_PRECISION_BF16) { dan_set_error("unknown precision %d", precision); return DAN_E_INVALID; }
  if (precision == DAN_PRECISION_BF16 && !dan_bf16_supported(m)) {
    dan_set_error("bf16 tcgen05 path does not cover this configuration: %s", dan_bf16_unsupported_reason(m));
    return DAN_E_UNSUPPORTED;
  }
  return DAN_OK;
}

int dan_forward(dan_model* m, int precision, const uint8_t* reads, const uint8_t* q_scores, const uint8_t* strands,
                const uint8_t* ref, const uint8_t* ref_masks, const uint8_t* var_masks, int batch, float* heads_out,
                void* workspace, size_t workspace_bytes, void* stream) {
  g_launches = 0;
  int rc = check_forward_args(m, precision, reads, q_scores, strands, ref, ref_masks, var_masks, batch, heads_out);
  if (rc) return rc;
  if (batch == 0) return DAN_OK;
  if (!workspace) { dan_set_error("null workspace"); return DAN_E_WORKSPACE; }
  DevInputs in{reads, q_scores, strands, ref, ref_masks, var_masks};
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (precision == DAN_PRECISION_BF16) return dan_bf16_forward(m, in, batch, heads_out, workspace, workspace_bytes, st);
  return dan_fp32_forward(m, in, batch, heads_out, workspace, workspace_bytes, st);
}

// ---- host-buffer entry point: chunked, double-buffered H2D staging on a side stream (north_star item 4) -------------------
// The batch is cut into chunks of host_chunk() candidates. Chunk k+1 is copied from the caller's (pinned) host buffers into staging
// buffer (k+1)&1 on the model's copy stream while chunk k runs on the caller's stream; events order copy -> compute and
// compute -> reuse of the staging buffer. Only the first chunk's copy is exposed.
static const int kHostFirst = 128;
// staging chunk = the FC trunk's chunk (bf16: a whole number of conv-stack passes, ~1024 candidates; the 151 MB FC1 weight stream is read once per chunk either way)
static int host_chunk(const dan_model* m, int batch, int precision) {
  const int full = precision == DAN_PRECISION_BF16 ? dan_bf16_fc_chunk(m) : 1024;
  return batch < full ? (batch > 0 ? batch : 1) : full;
}
static size_t host_stage_bytes_chunk(const dan_model* m, int chunk) {
  const size_t tile = (size_t)chunk * m->P * m->R, vec = (size_t)chunk * m->P;
  return 3 * round_up_z(tile, 256) + 3 * round_up_z(vec, 256);
}

size_t dan_workspace_bytes_host(const dan_model* m, int batch, int precision) {
  if (!m || batch < 0) return 0;
  const int chunk = host_chunk(m, batch, precision);
  return round_up_z(dan_workspace_bytes(m, chunk, precision), 256) + 2 * host_stage_bytes_chunk(m, chunk) +
         round_up_z((size_t)(batch > 0 ? batch : 1) * DAN_NUM_HEAD_OUTPUTS * 4, 256);
}

int dan_forward_host(dan_model* m, int precision, const uint8_t* reads, const uint8_t* q_scores, const uint8_t* strands,
                     const uint8_t* ref, const uint8_t* ref_masks, const uint8_t* var_masks, int batch,
                     float* heads_out_host, void* workspace, size_t workspace_bytes, void* stream) {
  g_launches = 0;
  int rc = check_forward_args(m, precision, reads, q_scores, strands, ref, ref_masks, var_masks, batch, heads_out_host);
  if (rc) return rc;
  if (batch == 0) return DAN_OK;
  const int chunk = host_chunk(m, batch, precision);
  const size_t core = round_up_z(dan_workspace_bytes(m, chunk, precision), 256);
  const size_t stage_b = host_stage_bytes_chunk(m, chunk);
  if (!workspace || workspace_bytes < dan_workspace_bytes_host(m, batch, precision)) { dan_set_error("workspace too small for host staging"); return DAN_E_WORKSPACE; }
  std::lock_guard<std::mutex> lk(*m->host_mu);          // the copy stream and its events belong to the model handle
  if (!m->copy_stream) {
    DAN_CUDA_TRY(cudaStreamCreateWithFlags(&m->copy_stream, cudaStreamNonBlocking));
    for (int i = 0; i < 2; ++i) {
      DAN_CUDA_TRY(cudaEventCreateWithFlags(&m->ev_copied[i], cudaEventDisableTiming));
      DAN_CUDA_TRY(cudaEventCreateWithFlags(&m->ev_done[i], cudaEventDisableTiming));
    }
    DAN_CUDA_TRY(cudaEventCreateWithFlags(&m->ev_entry, cudaEventDisableTiming));
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream), cs = m->copy_stream;
  char* base = static_cast<char*>(workspace);
  char* stage_base[2] = {base + core, base + core + stage_b};
  float* dheads = reinterpret_cast<float*>(base + core + 2 * stage_b);
  const size_t tile1 = (size_t)m->P * m->R, vec1 = (size_t)m->P;
  // staging buffers may still be read by work queued earlier on the caller's stream
  DAN_CUDA_TRY(cudaEventRecord(m->ev_entry, st));
  DAN_CUDA_TRY(cudaStreamWaitEvent(cs, m->ev_entry, 0));
  // the first chunk is small (its copy is the only one that is not hidden), the rest are full FC-sized chunks
  const int first = batch > 2 * kHostFirst ? kHostFirst : chunk;
  int launches = 0;
  for (int k = 0, c0 = 0; c0 < batch; ++k) {
    const int want = k == 0 ? first : chunk, nb = batch - c0 < want ? batch - c0 : want, b = k & 1;
    if (k >= 2) DAN_CUDA_TRY(cudaStreamWaitEvent(cs, m->ev_done[b], 0));          // chunk k-2 has finished with this staging buffer
    char* p = stage_base[b];
    auto stage = [&](const uint8_t* src, size_t per_cand) -> const uint8_t* {
      uint8_t* d = reinterpret_cast<uint8_t*>(p);
      p += round_up_z((size_t)chunk * per_cand, 256);
      if (!src) return nullptr;
      cudaMemcpyAsync(d, src + (size_t)c0 * per_cand, (size_t)nb * per_cand, cudaMemcpyHostToDevice, cs);
      return d;
    };
    DevInputs in{};
    in.reads = stage(reads, tile1); in.q = stage(q_scores, tile1); in.strands = stage(strands, tile1);
    in.ref = stage(ref, vec1); in.ref_masks = stage(ref_masks, vec1); in.var_masks = stage(var_masks, vec1);
    DAN_CUDA_TRY(cudaGetLastError());
    DAN_CUDA_TRY(cudaEventRecord(m->ev_copied[b], cs));
    DAN_CUDA_TRY(cudaStreamWaitEvent(st, m->ev_copied[b], 0));
    float* out = dheads + (size_t)c0 * DAN_NUM_HEAD_OUTPUTS;
    g_launches = 0;
    if (precision == DAN_PRECISION_BF16) rc = dan_bf16_forward(m, in, nb, out, workspace, core, st);
    else rc = dan_fp32_forward(m, in, nb, out, workspace, core, st);
    if (rc) return rc;
    launches += g_launches;
    DAN_CUDA_TRY(cudaEventRecord(m->ev_done[b], st));
    c0 += nb;
  }
  g_launches = launches;
  DAN_CUDA_TRY(cudaMemcpyAsync(heads_out_host, dheads, (size_t)batch * DAN_NUM_HEAD_OUTPUTS * 4, cudaMemcpyDeviceToHost, st));
  return DAN_OK;
}

int dan_encode(dan_model* m, const uint8_t* reads, const uint8_t* q_scores, const uint8_t* strands, const uint8_t* ref,
               const uint8_t* ref_masks, const uint8_t* var_masks, int batch, float* x0_out, void* stream) {
  int rc = check_forward_args(m, DAN_PRECISION_FP32, reads, q_scores, strands, ref, ref_masks, var_masks, batch, x0_out);
  if (rc) return rc;
  if (batch == 0) return DAN_OK;
  DevInputs in{reads, q_scores, strands, ref, ref_masks, var_masks};
  return dan_fp32_encode_reference_order(m, in, batch, x0_out, static_cast<cudaStream_t>(stream));
}

int dan_encode_bf16(dan_model* m, const uint8_t* reads, const uint8_t* q_scores, const uint8_t* strands, const uint8_t* ref,
                    const uint8_t* ref_masks, const uint8_t* var_masks, int batch, float* x0_out, void* stream) {
  int rc = check_forward_args(m, DAN_PRECISION_BF16, reads, q_scores, strands, ref, ref_masks, var_masks, batch, x0_out);
  if (rc) return rc;
  if (batch == 0) return DAN_OK;
  DevInputs in{reads, q_scores, strands, ref, ref_masks, var_masks};
  return dan_bf16_encode_reference_order(m, in, batch, x0_out, static_cast<cudaStream_t>(stream));
}

size_t dan_train_tape_bytes(const dan_model* m, int batch) {
  if (!m || batch < 1) return 0;
  if (const char* why = dan_train_unsupported_reason(m)) {
    dan_set_error("training kernels do not cover this configuration: %s", why);
    return 0;
  }
  return dan_train_tape_bytes_impl(m, batch);
}

static int check_train_args(dan_model* m, const dan_weights* params, const uint8_t* reads, const uint8_t* q, const uint8_t* s, const uint8_t* ref,
                            const uint8_t* rm, const uint8_t* vm, int batch, const void* out, float dropout_p) {
  int rc = check_forward_args(m, DAN_PRECISION_FP32, reads, q, s, ref, rm, vm, batch, out);
  if (rc) return rc;
  if (!params) { dan_set_error("null parameter struct"); return DAN_E_INVALID; }
  if (batch < 1) { dan_set_error("training needs at least one candidate"); return DAN_E_INVALID; }
  if (!(dropout_p >= 0.f && dropout_p < 1.f)) { dan_set_error("dropout probability %g outside [0, 1)", dropout_p); return DAN_E_INVALID; }
  if (const char* why = dan_train_unsupported_reason(m)) { dan_set_error("training kernels do not cover this configuration: %s", why); return DAN_E_UNSUPPORTED; }
  for (int l = 0; l < m->L; ++l)
    if (m->cfg.use_batchnorm && (!params->bn_w[l] || !params->bn_b[l] || !params->bn_mean[l] || !params->bn_var[l])) { dan_set_error("missing BatchNorm tensors of layer %d", l + 1); return DAN_E_INVALID; }
  if (m->cfg.pool_combine_dimension > 0 && (!params->post_pool_w || !params->post_pool_b)) { dan_set_error("missing post_pool_w / post_pool_b"); return DAN_E_INVALID; }
  return DAN_OK;
}

int dan_train_forward(dan_model* m, const dan_weights* params, const uint8_t* reads, const uint8_t* q_scores, const uint8_t* strands,
                      const uint8_t* ref, const uint8_t* ref_masks, const uint8_t* var_masks, const uint8_t* removed, int batch,
                      float dropout_p, uint64_t seed, float* heads_out, void* tape, size_t tape_bytes, void* stream) {
  g_launches = 0;
  int rc = check_train_args(m, params, reads, q_scores, strands, ref, ref_masks, var_masks, batch, heads_out, dropout_p);
  if (rc) return rc;
  if (!tape) { dan_set_error("null tape"); return DAN_E_WORKSPACE; }
  DevInputs in{reads, q_scores, strands, ref, ref_masks, var_masks};
  return dan_train_forward_impl(m, params, in, removed, batch, dropout_p, seed, heads_out, tape, tape_bytes, static_cast<cudaStream_t>(stream));
}

int dan_backward(dan_model* m, const dan_weights* params, const uint8_t* reads, const uint8_t* q_scores, const uint8_t* strands,
                 const uint8_t* ref, const uint8_t* ref_masks, const uint8_t* var_masks, const uint8_t* removed, int batch,
                 float dropout_p, uint64_t seed, const float* dheads, const float* heads_out, const dan_weights* grads,
                 void* tape, size_t tape_bytes, void* stream) {
  g_launches = 0;
  int rc = check_train_args(m, params, reads, q_scores, strands, ref, ref_masks, var_masks, batch, heads_out, dropout_p);
  if (rc) return rc;
  if (!tape || !dheads || !grads) { dan_set_error("null tape / gradient pointer"); return DAN_E_INVALID; }
  if (m->cfg.pool_combine_dimension > 0 && (!grads->post_pool_w || !grads->post_pool_b)) { dan_set_error("missing post_pool_w / post_pool_b gradient tensors"); return DAN_E_INVALID; }
  DevInputs in{reads, q_scores, strands, ref, ref_masks, var_masks};
  return dan_backward_impl(m, params, in, removed, batch, dropout_p, seed, dheads, heads_out, grads, tape, tape_bytes, static_cast<cudaStream_t>(stream));
}

namespace {
// tools/format_vcf.py:107-138 per record; thresholds already resolved (dan_genotype_calls)
__global__ void dan_genotype_calls_kernel(const float4* __restrict__ scores, const int32_t* __restrict__ ref_len, const int32_t* __restrict__ var_len, int batch,
                                          dan_call_thresholds t, int8_t* __restrict__ gt_out, int32_t* __restrict__ q_out) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= batch) return;
  const float4 s = scores[b];
  // the script thresholds the "%.8f" text of the scores parsed back to double (utils.py:171-176, format_vcf.py:108)
  const double nv = rint((double)s.y * 1e8) / 1e8, ov = rint((double)s.w * 1e8) / 1e8;
  const int rl = ref_len[b], vl = var_len[b];
  const bool snp = rl == 1 && vl == 1, lng = rl >= 3 || vl >= 3, del = rl > 1 && vl == 1;
  const double thr = snp ? t.snp : (lng ? t.long_indel : (del ? t.del : t.indel));
  const double hz = snp ? t.snp_zygo : (lng ? t.long_indel_zygo : (del ? t.del_zygo : t.indel_zygo));
  const double margin = (1.0 - nv) - thr;
  if (margin >= 0.0) {
    gt_out[b] = ov >= hz ? 2 : 1;
    q_out[b] = (int)(margin / (1.0 - thr) * 50.0);      // SCORE_BUCKETS, format_vcf.py:42,136-137
  } else {
    gt_out[b] = 0;
    q_out[b] = -1;
  }
}
}  // namespace

int dan_genotype_calls(const float* scores, const int32_t* ref_len, const int32_t* var_len, int batch, const dan_call_thresholds* thr,
                       int8_t* gt_out, int32_t* q_out, void* stream) {
  if (batch < 0 || !thr || (batch > 0 && (!scores || !ref_len || !var_len || !gt_out || !q_out))) { dan_set_error("dan_genotype_calls: bad arguments"); return DAN_E_INVALID; }
  if (batch == 0) return DAN_OK;
  dan_call_thresholds t = *thr;                         // format_vcf.py:57-80
  if (!(t.indel > 0.0)) { t.indel = t.snp; t.indel_zygo = t.snp_zygo; t.long_indel = t.indel; t.long_indel_zygo = t.indel_zygo; t.del = t.indel; t.del_zygo = t.indel_zygo; }
  else {
    if (!(t.long_indel > 0.0)) { t.long_indel = t.indel; t.long_indel_zygo = t.indel_zygo; }
    if (!(t.del > 0.0)) { t.del = t.indel; t.del_zygo = t.indel_zygo; }
  }
  dan_genotype_calls_kernel<<<(batch + 255) / 256, 256, 0, static_cast<cudaStream_t>(stream)>>>(reinterpret_cast<const float4*>(scores), ref_len, var_len, batch, t, gt_out, q_out);
  DAN_CUDA_TRY(cudaGetLastError());
  return DAN_OK;
}

namespace {
// 8 independent FFMA chains per thread, 4096 FFMAs per chain and call
__global__ void __launch_bounds__(256) fma_peak_kernel(float* __restrict__ sink, int reps) {
  float a[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) a[i] = (float)(threadIdx.x + i) * 1e-3f;
  const float m = 1.0000001f, c = 1e-7f;
  for (int r = 0; r < reps; ++r) {
#pragma unroll
    for (int k = 0; k < 512; ++k) {
#pragma unroll
      for (int i = 0; i < 8; ++i) a[i] = fmaf(a[i], m, c);
    }
  }
  float t = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) t += a[i];
  if (t == 12345.678f) sink[0] = t;
}
}  // namespace

double dan_measure_fma_tflops(double ms, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int dev = 0, sms = 0;
  float* sink = nullptr;
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  double result = -1.0;
  if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return -1.0;
  if (cudaMalloc(&sink, 4) != cudaSuccess) return -1.0;
  if (cudaEventCreate(&e0) == cudaSuccess && cudaEventCreate(&e1) == cudaSuccess) {
    const int blocks = sms * 8;
    auto run = [&](int reps) -> double {
      cudaEventRecord(e0, st);
      fma_peak_kernel<<<blocks, 256, 0, st>>>(sink, reps);
      cudaEventRecord(e1, st);
      if (cudaEventSynchronize(e1) != cudaSuccess) return -1.0;
      float t = 0.f;
      cudaEventElapsedTime(&t, e0, e1);
      return (double)t;
    };
    const double flop_per_rep = 2.0 * 8 * 512 * 256.0 * blocks;
    double t = run(8);                                     // warm-up and calibration
    if (t > 0.0) {
      int reps = (int)(8.0 * (ms > 1.0 ? ms : 1.0) / t) + 1;
      if (reps > 1 << 20) reps = 1 << 20;
      t = run(reps);
      if (t > 0.0) result = flop_per_rep * reps / (t * 1e-3) / 1e12;
    }
  }
  if (e0) cudaEventDestroy(e0);
  if (e1) cudaEventDestroy(e1);
  cudaFree(sink);
  return result;
}

int dan_scores(const float* heads, int batch, float* scores_out, void* stream) {
  if (batch < 0) { dan_set_error("negative batch"); return DAN_E_INVALID; }
  if (batch == 0) return DAN_OK;
  if (!heads || !scores_out) { dan_set_error("heads / scores pointer is null"); return DAN_E_INVALID; }
  if (reinterpret_cast<uintptr_t>(scores_out) & 15) { dan_set_error("scores_out must be 16-byte aligned"); return DAN_E_INVALID; }
  dan_scores_kernel<<<(batch + 255) / 256, 256, 0, static_cast<cudaStream_t>(stream)>>>(heads, batch, reinterpret_cast<float4*>(scores_out));
  dan_count_launch(1);
  DAN_CUDA_TRY(cudaGetLastError());
  return DAN_OK;
}

int dan_make_mask_vectors(const char* const* ref_alleles, const char* const* var_alleles, const uint8_t* references, int n,
                          uint8_t* ref_masks, uint8_t* var_masks, int32_t* status) {
  if (n < 0) { dan_set_error("negative record count"); return DAN_E_INVALID; }
  if (n == 0) return DAN_OK;
  if (!ref_alleles || !var_alleles || !references || !ref_masks || !var_masks) { dan_set_error("null pointer"); return DAN_E_INVALID; }
  int failed = 0, first = -1, first_code = 0;
  for (int i = 0; i < n; ++i) {
    uint8_t* rm = ref_masks + (size_t)i * DAN_MASK_READ_LEN;
    uint8_t* vm = var_masks + (size_t)i * DAN_MASK_READ_LEN;
    memset(rm, 0, DAN_MASK_READ_LEN); memset(vm, 0, DAN_MASK_READ_LEN);
    int code = (ref_alleles[i] && var_alleles[i]) ? mask_one(ref_alleles[i], var_alleles[i], references + (size_t)i * DAN_MASK_READ_LEN, rm, vm)
                                                  : (int)DAN_MASK_E_ALLELE_CHAR;
    if (code != DAN_MASK_OK) {
      memset(rm, 0, DAN_MASK_READ_LEN); memset(vm, 0, DAN_MASK_READ_LEN);
      if (!failed) { first = i; first_code = code; }
      ++failed;
    }
    if (status) status[i] = code;
  }
  if (failed) { dan_set_error("%d of %d records could not be decoded (first: record %d, DAN_MASK_E code %d)", failed, n, first, first_code); return DAN_E_INVALID; }
  return DAN_OK;
}

int dan_format_vcf_info(const float* scores, int n, char* out, size_t out_bytes) {
  if (n < 0) { dan_set_error("negative record count"); return DAN_E_INVALID; }
  if (n == 0) return DAN_OK;
  if (!scores || !out) { dan_set_error("scores / out pointer is null"); return DAN_E_INVALID; }
  if (out_bytes < (size_t)n * DAN_VCF_INFO_STRIDE) { dan_set_error("output buffer too small: need %zu bytes", (size_t)n * DAN_VCF_INFO_STRIDE); return DAN_E_INVALID; }
  for (int i = 0; i < n; ++i) {
    const float* s4 = scores + (size_t)i * DAN_NUM_SCORE_OUTPUTS;
    for (int j = 0; j < 4; ++j)
      if (!(s4[j] >= 0.f && s4[j] <= 1.f)) { dan_set_error("score %d of record %d is not a probability", j, i); return DAN_E_INVALID; }
    // python's '%.8f' % float32 widens to double first (utils.py:171-176); printf rounds the same way (correctly rounded decimal)
    snprintf(out + (size_t)i * DAN_VCF_INFO_STRIDE, DAN_VCF_INFO_STRIDE, "BP=%.8f;NV=%.8f;HV=%.8f;OV=%.8f",
             (double)s4[0], (double)s4[1], (double)s4[2], (double)s4[3]);
  }
  return DAN_OK;
}

int dan_debug_fc_input(dan_model* m, int precision, int batch, const void* workspace, float* out, void* stream) {
  if (!m || !workspace || !out || batch < 1) { dan_set_error("bad argument"); return DAN_E_INVALID; }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (precision == DAN_PRECISION_BF16) return dan_bf16_debug_fc_input(m, batch, workspace, out, st);
  return dan_fp32_debug_fc_input(m, batch, workspace, out, st);
}

}  // extern "C"
