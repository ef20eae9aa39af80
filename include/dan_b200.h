/* dan_b200.h — C-ABI of the B200-native DAN ("Basic2DNet") forward path.
 *
 * The reference has no FFI layer: its boundary for this path is the Python module interface of
 * dl4vc/model.py (class Basic2DNet, reference dl4vc/model.py:31-961). Each entry point below is what a binding
 * for that interface has to reach; the citation says which reference lines it replaces. dl4vc_b200/model.py is the
 * ctypes binding shipped with this repo (INTEGRATION.md shows the three-line overlay for the reference tree).
 *
 * Conventions: plain pointers and sizes only (no torch types); every function returns 0 on success or a negative
 * DAN_E_* code, with a thread-local message available from dan_last_error(); nothing calls exit(). All device
 * pointers must belong to the CUDA device that was current when the model handle was created. Functions taking a
 * stream are asynchronous with respect to the host and re-entrant per (model, stream) pair as long as each
 * concurrent call uses its own workspace.
 */
#ifndef DAN_B200_H
#define DAN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DAN_MAX_LAYERS 12
#define DAN_MAX_FC 4
#define DAN_NUM_HEAD_OUTPUTS 27 /* xbinary(2) xVT(3) xAF(1) xCov(1) xVB(10) xVR(10): dl4vc/model.py:919-921,953-958 */

enum { DAN_OK = 0, DAN_E_INVALID = -1, DAN_E_UNSUPPORTED = -2, DAN_E_CUDA = -3, DAN_E_WORKSPACE = -4 };

/* arithmetic of the contraction kernels */
enum {
  DAN_PRECISION_FP32 = 0, /* CUDA-core FFMA, fp32 storage: logits within 1e-4 relative of the reference */
  DAN_PRECISION_BF16 = 1  /* tcgen05 tensor cores, bf16 operands, fp32 accumulation in TMEM */
};

/* Shape of the network = the constructor arguments of Basic2DNet that change arithmetic
 * (dl4vc/model.py:35-53; PROD values = call_variants.sh:101-147). */
typedef struct dan_config {
  int32_t total_conv_layers;            /* model.py:45  */
  int32_t channels;                     /* init_conv_channels == final_conv_channels, model.py:36 */
  int32_t embed_dim;                    /* model.py:36 (20) */
  int32_t use_q_scores;                 /* model.py:38 */
  int32_t use_strands;                  /* model.py:38 */
  int32_t use_reads_ref_var_mask;       /* model.py:40 */
  int32_t dilation[DAN_MAX_LAYERS];     /* per layer, model.py:213-229 */
  int32_t is_residual[DAN_MAX_LAYERS];  /* model.py:246 */
  int32_t pool_after[DAN_MAX_LAYERS];   /* 1: read-mean of this layer's output is added to the next layer's input, model.py:734-742,766-772 */
  int32_t use_batchnorm;                /* model.py:49 */
  int32_t highway;                      /* append_bottleneck_highway_reads, model.py:43 */
  int32_t bottleneck;                   /* bottleneck_channels == bottleneck_linear_outputs, model.py:42 */
  int32_t concat_hw_reads;              /* model.py:43 */
  int32_t pool_combine_dimension;       /* model.py:51 */
  int32_t skip_final_maxpool;           /* model.py:51 */
  int32_t num_fc;                       /* len(layer_sizes), model.py:35 */
  int32_t fc_sizes[DAN_MAX_FC];
  int32_t num_reads;                    /* 100, model.py:41 / dataset.py:398 */
  int32_t read_len;                     /* 201, model.py:41 */
} dan_config;

/* fp32 parameter tensors in the reference's state_dict layout (SURVEY App. B), DEVICE pointers.
 * Unused entries (layers beyond total_conv_layers, disabled features) are NULL. */
typedef struct dan_weights {
  const float* embeddings;                      /* (10, embed_dim)                 embeddings.weight */
  const float* pe;                              /* (read_len, embed_dim)           pe[0] */
  const float* conv_w[DAN_MAX_LAYERS];          /* (C, Cin, 1, 3)                  conv1D_layers.l.weight */
  const float* conv_b[DAN_MAX_LAYERS];          /* (C)                                                        */
  const float* bn_w[DAN_MAX_LAYERS];            /* (C) gamma                       bn1D_layers.l.weight */
  const float* bn_b[DAN_MAX_LAYERS];            /* (C) beta */
  const float* bn_mean[DAN_MAX_LAYERS];         /* (C) running_mean */
  const float* bn_var[DAN_MAX_LAYERS];          /* (C) running_var */
  const float* res_w[DAN_MAX_LAYERS];           /* (C, C, 1, 1) indexed by LAYER (0-based), NULL if not residual */
  const float* res_b[DAN_MAX_LAYERS];
  const float* bott_w[DAN_MAX_LAYERS];          /* (bott, C, 1, 1)                 conv1D_bottleneck_layers.l */
  const float* bott_b[DAN_MAX_LAYERS];
  const float* comp_w[DAN_MAX_LAYERS];          /* (bott, bott, 1, read_len)       conv1D_compression_layers.l */
  const float* comp_b[DAN_MAX_LAYERS];
  const float* post_pool_w;                     /* (pool_combine_dimension, pooled_features) */
  const float* post_pool_b;
  const float* fc_w[DAN_MAX_FC];                /* (out, in)                       conv2hidden.{1,4}.weight */
  const float* fc_b[DAN_MAX_FC];
  const float* head_w;                          /* (27, hidden) rows in DAN_NUM_HEAD_OUTPUTS order */
  const float* head_b;                          /* (27) */
} dan_weights;

typedef struct dan_model dan_model; /* opaque: config + packed device weights */

/* Thread-local text of the last error raised by this library on the calling thread. */
const char* dan_last_error(void);
/* Library build identification: "dan_b200 <version> sm_100a". */
const char* dan_version(void);

/* Replaces Basic2DNet.__init__ (dl4vc/model.py:35-432): validates the configuration and allocates the packed
 * weight store on the current CUDA device. DAN_E_UNSUPPORTED for shapes the kernels do not cover. */
int dan_model_create(const dan_config* cfg, dan_model** out);
int dan_model_destroy(dan_model* m);

/* Replaces load_state_dict / .cuda() (main.py:117,124): folds BatchNorm running statistics into scale/shift,
 * re-lays every matrix for the kernels (fp32 K-major and bf16 UMMA core-matrix order). Must be called again
 * whenever parameters change. Asynchronous on `stream`. */
int dan_model_load_weights(dan_model* m, const dan_weights* w, void* stream);

/* Number of candidates the conv stack processes per internal pass (activations of one pass stay L2-resident). */
int dan_model_set_pass_candidates(dan_model* m, int candidates);

/* Test hook: behaviour switches of a model handle. DAN_FLAG_LAYERWISE makes the bf16 path run its layer-by-layer kernels (the
 * route of the configurations the fused conv-stack kernel does not take) on every configuration, so that both routes can be
 * compared on the same inputs. */
enum { DAN_FLAG_LAYERWISE = 1 };
int dan_model_set_flags(dan_model* m, int flags);

/* Test hook: which route dan_forward takes at DAN_PRECISION_BF16 with the handle's current flags. 0: the bf16 path does not cover the
 * configuration (dan_forward returns DAN_E_UNSUPPORTED naming the reason), 1: the fused conv-stack kernel (dan_stack.cuh), 2: layer by
 * layer (dan_layerwise.cuh). */
enum { DAN_BF16_ROUTE_NONE = 0, DAN_BF16_ROUTE_FUSED = 1, DAN_BF16_ROUTE_LAYERWISE = 2 };
int dan_model_bf16_route(const dan_model* m);

/* Bytes of device scratch dan_forward needs for a batch of `batch` candidates at `precision`. */
size_t dan_workspace_bytes(const dan_model* m, int batch, int precision);

/* Replaces Basic2DNet.forward in eval mode (dl4vc/model.py:434-961) for a batch of `batch` candidates.
 * Inputs are the loader's tensors narrowed to uint8, DEVICE pointers, layout [batch][position][read]
 * (dl4vc/dataset.py:672-680): reads, q_scores, strands are batch*read_len*num_reads bytes; ref, ref_masks,
 * var_masks are batch*read_len bytes. q_scores / strands / masks may be NULL when the config does not use them.
 * heads_out: batch*27 fp32, row = [xbinary(2) xVT(3) sigmoid(xAF) leaky_relu(xCov) xVB(10) xVR(10)]. */
int dan_forward(dan_model* m, int precision, const uint8_t* reads, const uint8_t* q_scores,
                const uint8_t* strands, const uint8_t* ref, const uint8_t* ref_masks, const uint8_t* var_masks,
                int batch, float* heads_out, void* workspace, size_t workspace_bytes, void* stream);

/* Same contract with HOST buffers (pinned for true asynchrony): stages the uint8 inputs to the device on
 * `stream`, runs dan_forward and copies the batch*27 fp32 results back. Staging memory is taken from the tail of
 * the workspace (dan_workspace_bytes_host). This is the call the end-to-end benchmark times. */
size_t dan_workspace_bytes_host(const dan_model* m, int batch, int precision);
int dan_forward_host(dan_model* m, int precision, const uint8_t* reads, const uint8_t* q_scores,
                     const uint8_t* strands, const uint8_t* ref, const uint8_t* ref_masks,
                     const uint8_t* var_masks, int batch, float* heads_out_host, void* workspace,
                     size_t workspace_bytes, void* stream);

/* Replaces the caller-side score post-ops of trainer.test (dl4vc/trainer.py:611-623, use_var_type_threshold off) on the
 * device, so that only 4 floats per candidate have to cross PCIe when the caller writes VCF records:
 * scores_out[b] = { 1 - softmax(xbinary)[0],  softmax(xVT)[0], softmax(xVT)[1], softmax(xVT)[2] }
 * (variant score, P{no variant}, P{het}, P{hom}; the BP / NV / HV / OV fields of dl4vc/utils.py:162-178).
 * heads: batch*27 fp32 as written by dan_forward, scores_out: batch*4 fp32, both DEVICE pointers. */
#define DAN_NUM_SCORE_OUTPUTS 4
int dan_scores(const float* heads, int batch, float* scores_out, void* stream);

/* Replaces the per-record thresholding of tools/format_vcf.py (filter_format_vcf, :107-138) for a batch, on the device, so that a caller
 * can drop the records that will not be written before their scores cross PCIe. For candidate b with scores row
 * { BP, NV, HV, OV } (dan_scores) and allele lengths ref_len[b] / var_len[b] (the REF / ALT columns of its VCF record):
 *   class: SNP (1/1), long indel (either allele >= 3 bases), short delete (ref > 1, alt == 1), other indel; the class picks the
 *   call threshold and the homozygous threshold;  margin = (1 - NV) - threshold;  margin < 0 -> gt_out[b] = 0, q_out[b] = -1;
 *   else gt_out[b] = 2 ("1/1") if OV >= homozygous threshold else 1 ("0/1"), q_out[b] = int(margin / (1 - threshold) * 50).
 * NV and OV are first rounded to 8 decimals, the values the script parses back from the "%.8f" text of utils.py:171-176, and the
 * arithmetic is double like Python's, so the integers match the script's. Thresholds are the script's command-line values;
 * non-positive indel / long-indel / delete call thresholds fall back as format_vcf.py:57-80 does (long indel -> indel -> SNP; the script
 * leaves the delete threshold unassigned when --indel_threshold is not given and raises on the first short delete: here it falls back
 * to the indel pair). The script's merge of several records at one position (:150-215) works on sorted text and stays with the caller.
 * scores, ref_len, var_len, gt_out, q_out: DEVICE pointers. */
typedef struct dan_call_thresholds {
  double snp, snp_zygo, indel, indel_zygo, long_indel, long_indel_zygo, del, del_zygo;
} dan_call_thresholds;
int dan_genotype_calls(const float* scores, const int32_t* ref_len, const int32_t* var_len, int batch, const dan_call_thresholds* thr,
                       int8_t* gt_out, int32_t* q_out, void* stream);

/* Replaces the per-record string formatting of utils.append_vcf_records (dl4vc/utils.py:171-176) for a batch: for each of the n
 * rows of `scores` (HOST pointer, n*4 fp32 as written by dan_scores) writes the fixed-width, NUL-terminated text
 * "BP=%.8f;NV=%.8f;HV=%.8f;OV=%.8f" at out + i*DAN_VCF_INFO_STRIDE (HOST buffer of n*DAN_VCF_INFO_STRIDE bytes). Values are
 * probabilities in [0, 1], so every field is 10 characters and a record is 55 characters + NUL. Pure host code (no CUDA call). */
#define DAN_VCF_INFO_STRIDE 56
int dan_format_vcf_info(const float* scores, int n, char* out, size_t out_bytes);

/* Replaces the loader's per-item proposal-mask decode, get_read_mask_vectors + simple_variant_encoding_vectors
 * (dl4vc/dataset.py:86-250), for a batch of n records: ref_alleles[i] / var_alleles[i] are the REF / ALT columns of the VCF record
 * (NUL-terminated), references + i*201 the encoded 201-column reference window of the pileup (base_enum codes, '-' = 5).
 * Writes ref_masks / var_masks (n*201 bytes each, HOST pointers): 0 everywhere except the allele's bases starting at the
 * window's centre column (rewound past insert-gap columns), with the reference's conventions — deletes padded with '-' (5) in
 * the variant mask, inserts with 'noinsert' (8) in the reference mask, ALT clipped to 51 bases, gap columns inside a deleted
 * stretch left as "don't care" (0). status[i] (may be NULL) is 0 or the reason the reference itself would have raised for the
 * record (DAN_MASK_E_*); masks of a failed record are all zero. Returns DAN_OK when every record decoded, DAN_E_INVALID otherwise.
 * Pure host code (no CUDA call). */
enum { DAN_MASK_OK = 0, DAN_MASK_E_ALLELE_CHAR = 1,   /* character outside base_enum (KeyError) */
       DAN_MASK_E_UNSUPPORTED = 2,                   /* neither SNP (both alleles in "AaTtCcG"), delete nor insert: equal lengths (UnboundLocalError) */
       DAN_MASK_E_SHAPE = 3,                         /* delete with ALT longer than one base / insert with REF longer than one base (assert) */
       DAN_MASK_E_REF_MISMATCH = 4,                  /* window does not hold the record's reference bases (assert) */
       DAN_MASK_E_WINDOW = 5 };                      /* allele runs past the window (ValueError) or no base at or before the centre */
#define DAN_MASK_READ_LEN 201
int dan_make_mask_vectors(const char* const* ref_alleles, const char* const* var_alleles, const uint8_t* references, int n,
                          uint8_t* ref_masks, uint8_t* var_masks, int32_t* status);

/* ---- training (BASELINE configs[4]) -----------------------------------------------------------------------------------------
 * Replaces Basic2DNet.forward with self.training set and the autograd graph PyTorch builds behind it (dl4vc/model.py:434-961 called
 * from dl4vc/trainer.py:213-217; backward at trainer.py:426-439). fp32 on the CUDA-core kernels of the accuracy path.
 *
 * dan_train_forward: like dan_forward (DEVICE uint8 inputs, batch*27 fp32 outputs) but BatchNorm normalises with the statistics of
 * this batch and updates the running statistics IN PLACE through params->bn_mean / bn_var (momentum 0.1, unbiased variance), the
 * three Dropout modules of the FC trunk use a counter-based mask derived from (seed, element index) with probability dropout_p, and
 * reads flagged in `removed` (batch*num_reads bytes, may be NULL) are replaced by the empty-read encoding (the read-removal
 * augmentation of model.py:633-716; the caller picks the reads like the reference's randperm does). `params` are the live fp32
 * parameter tensors (state_dict layout); dan_model_load_weights must have been called on the same values. Everything the backward
 * pass needs stays in `tape` (dan_train_tape_bytes).
 *
 * dan_backward: d(loss)/d(heads) (batch*27, w.r.t. the returned, activated outputs) -> gradient of every parameter tensor, written
 * (not accumulated) into the tensors `grads` points to (same layout as `params`; head_w / head_b as the 27-row concatenation;
 * embeddings may be NULL to skip the embedding table; post_pool_w / post_pool_b are required, in params and in grads, when
 * pool_combine_dimension > 0). Must follow dan_train_forward on the same tape, inputs, seed and dropout_p. */
size_t dan_train_tape_bytes(const dan_model* m, int batch);
int dan_train_forward(dan_model* m, const dan_weights* params, const uint8_t* reads, const uint8_t* q_scores, const uint8_t* strands,
                      const uint8_t* ref, const uint8_t* ref_masks, const uint8_t* var_masks, const uint8_t* removed, int batch,
                      float dropout_p, uint64_t seed, float* heads_out, void* tape, size_t tape_bytes, void* stream);
int dan_backward(dan_model* m, const dan_weights* params, const uint8_t* reads, const uint8_t* q_scores, const uint8_t* strands,
                 const uint8_t* ref, const uint8_t* ref_masks, const uint8_t* var_masks, const uint8_t* removed, int batch,
                 float dropout_p, uint64_t seed, const float* dheads, const float* heads_out, const dan_weights* grads,
                 void* tape, size_t tape_bytes, void* stream);

/* Replaces the trainer's per-step loss block (dl4vc/trainer.py:252-255,309-313,426-427; dl4vc/objectives.py:49-112) and the host round
 * trips around it (trainer.py:258,263,267) with one kernel: heads (batch*27 fp32 as returned by dan_train_forward) + targets (all DEVICE
 * pointers: label<=1, var_type, allele_freq, coverage * 0.01, var_base_enum, var_ref_enum, per-example weight or NULL) ->
 *   losses_out[8] = { binary, genotype, allele-frequency, coverage, variant-base, reference-base, weighted total, number of close
 *                     (easy) examples }, dheads_out = d(total)/d(heads) (batch*27, ready for dan_backward), close_vt / close_bin =
 *   the "well classified" flags of objectives.py:110-111 (batch bytes each). dan_close_table_update scatters flags into the per-example
 *   table the next epoch's sampler reads (dl4vc/dataset.py:480,719-732) without leaving the device. */
typedef struct dan_loss_config {
  float label_smoothing;      /* arguments.py:33 (train_variant_caller.sh: 0.001) */
  float close_match_window;   /* arguments.py:35 (2.0) */
  float focal_gamma;          /* arguments.py:37 (0.2) */
  float focal_alpha;          /* arguments.py:39 (1.0) */
  float fp_train_weight;      /* pos_weight[0] of both classification losses, trainer.py:84-96 */
  float binary_weight;        /* trainer.py:426 */
  float aux_weight;           /* args.auxillary_loss_weight */
  float aux_allele_weight;    /* args.auxillary_loss_allele_weight */
  float aux_bases_weight;     /* args.auxillary_loss_bases_weight */
} dan_loss_config;
int dan_losses(const float* heads, int batch, const int32_t* target_binary, const int32_t* target_var_type, const float* target_allele_freq,
               const float* target_coverage, const int32_t* target_var_base, const int32_t* target_ref_base, const float* example_weight,
               const dan_loss_config* cfg, float* losses_out, float* dheads_out, uint8_t* close_vt, uint8_t* close_bin, void* stream);
int dan_close_table_update(uint8_t* table, int64_t table_len, const int64_t* idx, const uint8_t* flags, int batch, void* stream);

/* Replaces the per-item Python loader, ContextDatasetFromNumpy._get_generator (dl4vc/dataset.py:500-680: row window, sample_single_reads
 * :256-287, parse_vcf utils.py:19-72, count_variants_from_single_reads :340-362, get_read_mask_vectors :112-250) for a batch of record
 * indices: `records` are raw records of the compound type tools/convert_bam_single_reads.py writes (:694-698; 123 965 bytes, no padding),
 * `record_stride` bytes apart (np.memmap of that dtype). Outputs are HOST pointers (pin them for dan_forward_host), [candidate][position]
 * [read] for the three tiles; any output except reads / ref / masks may be NULL. Pileups deeper than max_reads are reduced to a sorted
 * subset of their rows chosen from (seed, record index) — the reference draws it from the unseeded global numpy generator. status[i] is
 * DAN_REC_OK or the reason the reference's loader raises on the record; blacklist[i] = 1 where the reference catches the mask assertion
 * and substitutes all-pad masks. Pure host code. Returns DAN_E_INVALID if any record failed. */
#define DAN_RECORD_BYTES 123965
enum { DAN_REC_OK = 0, DAN_REC_E_VCF_FIELDS = 1, DAN_REC_E_ALLELE = 2, DAN_REC_E_UNKNOWN_MUTATION = 3, DAN_REC_E_VCF_INFO = 4, DAN_REC_E_MASK = 5 };
typedef struct dan_feeder_config {
  int32_t max_reads;          /* 100 (dataset.py:398) */
  int32_t store_max_reads;    /* 200 (rows of the stored pileup the window is taken from, dataset.py:410) */
  int32_t use_q_scores, use_strands;   /* args.model_use_q_scores / model_use_strands: unused tiles stay zero (dataset.py:563,577) */
  int32_t keep_candidate_af;  /* args.aux_keep_candidate_af (dataset.py:616) */
  uint64_t seed;
} dan_feeder_config;
typedef struct dan_record_batch {
  uint8_t *reads, *q_scores, *strands;          /* n * 201 * max_reads */
  uint8_t *ref, *ref_masks, *var_masks;         /* n * 201 */
  uint8_t* label; int32_t* num_reads; uint8_t* is_snp; int32_t* var_type; float* allele_freq; int32_t* coverage;
  int32_t *var_base_enum, *var_ref_enum; uint8_t* blacklist; int32_t* status;
} dan_record_batch;
int dan_decode_records(const void* records, size_t record_stride, const int64_t* indices, int n, const dan_feeder_config* cfg,
                       const dan_record_batch* out);

/* The decode in two passes. The header pass (host) does everything that is not tile bytes: row window and read sampling, VCF parse,
 * allele counts at the proposal column over the chosen rows, coverage / allele frequency, proposal masks, blacklist and status. The
 * tile pass gathers the chosen stored rows of single_reads / q-scores / strand into the [position][read] tiles. dan_decode_records
 * runs both on the host; dan_decode_records_device runs the tile pass on the device.
 * One header per record: tile column j (j < num_rows) is stored row rows[j] of the record; columns from num_rows on are zero.
 * ref_len / var_len are the lengths of the VCF record's REF / ALT columns (0 if it has too few columns). */
typedef struct dan_record_header {
  int32_t window_start;       /* first stored row of the window (dataset.py:517-521) */
  int32_t num_rows;           /* chosen rows = tile columns holding a read, <= max_reads */
  int32_t ref_len, var_len;
  uint8_t rows[200];          /* stored-row indices of tile columns 0 .. num_rows-1, ascending */
} dan_record_header;

/* Header pass alone (pure host code): same arguments as dan_decode_records; fills headers[n], the masks and the scalars of `out`
 * (its tile and ref pointers are not used). Returns DAN_E_INVALID if any record failed. */
int dan_decode_record_headers(const void* records, size_t record_stride, const int64_t* indices, int n, const dan_feeder_config* cfg,
                              const dan_record_batch* out, dan_record_header* headers);

/* ---- compressed record files ------------------------------------------------------------------------------------------------------
 * File layout (all fields little-endian; written and opened by dl4vc_b200/feeder.py):
 *   header, 64 bytes: magic "DL4VCZR1", u32 version = 1, u32 record_bytes = DAN_RECORD_BYTES, u64 count, u64 index_off,
 *                     u64 sidecar_off, u64 data_off, u64 data_bytes, u32 sidecar_bytes = DAN_SIDECAR_BYTES, u32 reserved = 0;
 *   index   at index_off:   count entries of 12 bytes, u64 offset into the data section + u32 compressed length;
 *   sidecar at sidecar_off: count sidecars of DAN_SIDECAR_BYTES (dan_record_sidecars);
 *   data    at data_off:    data_bytes of RFC 1950 zlib streams, one per record holding its DAN_RECORD_BYTES, in record order.
 * A sidecar holds exactly the record bytes the header pass reads, plus the name: [name 16][num_reads 4][label 1][vcfrec 128]
 * [ref_bases 201][single_reads column 100 of stored rows 0..199][column 101 of rows 0..199]. The header pass over a record's sidecar
 * gives the same headers, scalars and masks as over the record. */
#define DAN_SIDECAR_BYTES 750
int dan_record_sidecars(const void* records, size_t record_stride, int n, void* out);

/* dan_decode_record_headers over sidecars (DAN_SIDECAR_BYTES apart): sidecar indices[i] decodes into entry i, keyed by indices[i]. */
int dan_decode_sidecar_headers(const void* sidecars, const int64_t* indices, int n, const dan_feeder_config* cfg, const dan_record_batch* out,
                               dan_record_header* headers);

/* Batched zlib inflate on the device: stream i is src[offsets[i], offsets[i] + lengths[i]) and inflates into
 * dst[i * slot_bytes, (i + 1) * slot_bytes). Stored, fixed- and dynamic-Huffman blocks, 32 KB window, zlib header and Adler-32 trailer.
 * status[i] = DAN_INFLATE_OK only when the stream inflated to exactly slot_bytes and its Adler-32 matched; any other status leaves an
 * all-zero slot. Every read stays inside its stream and every write inside its slot, so a bad stream never affects another.
 * All pointers are DEVICE pointers; asynchronous on `stream`. */
enum { DAN_INFLATE_OK = 0, DAN_INFLATE_E_HEADER = 1, DAN_INFLATE_E_BLOCK = 2, DAN_INFLATE_E_CODES = 3, DAN_INFLATE_E_DISTANCE = 4,
       DAN_INFLATE_E_INPUT = 5, DAN_INFLATE_E_OUTPUT_LONG = 6, DAN_INFLATE_E_OUTPUT_SHORT = 7, DAN_INFLATE_E_ADLER = 8 };
int dan_inflate_device(const void* src, const uint64_t* offsets, const uint32_t* lengths, int n, void* dst, uint64_t slot_bytes,
                       int32_t* status, void* stream);

/* Batched zlib deflate on the device, the inverse of dan_inflate_device: input i is src[i * slot_bytes, (i + 1) * slot_bytes) and
 * becomes one complete RFC 1950 stream (2-byte header, deflate blocks, big-endian Adler-32) in dst[i * B, (i + 1) * B) with
 * B = dan_deflate_bound(slot_bytes) = slot_bytes + 5 * max(1, ceil(slot_bytes / 65535)) + 6, the size of the stored-block encoding (an
 * empty input still needs one block). lengths[i] receives the stream's length and status[i] DAN_DEFLATE_OK. The streams hold
 * dynamic-Huffman blocks, or stored blocks when those would be larger; no write leaves its slot. Distances stay within 32768 bytes and
 * the input, matches within 258 bytes. A stream's bytes depend only on its input: not on n, its position in the batch, the launch or
 * the device. All pointers are DEVICE pointers; asynchronous on `stream`. Before any launch: DAN_E_INVALID for n < 0 or a null
 * pointer, DAN_E_UNSUPPORTED for slot_bytes above DAN_DEFLATE_MAX_SLOT (the input must fit in one CTA's shared memory). n = 0
 * launches nothing. */
#define DAN_DEFLATE_MAX_SLOT 131072
enum { DAN_DEFLATE_OK = 0, DAN_DEFLATE_E_UNSUPPORTED = 1 };
size_t dan_deflate_bound(uint64_t slot_bytes);
int dan_deflate_device(const void* src, int n, uint64_t slot_bytes, void* dst, uint32_t* lengths, int32_t* status, void* stream);

/* Packs the n streams of dan_deflate_device back to back: offsets (DEVICE, n + 1 u64) receives the exclusive prefix sum of lengths
 * (offsets[n] = the total) and stream i moves from its slot in `slots` (stride dan_deflate_bound(slot_bytes)) to dst + offsets[i]. dst
 * (DEVICE) must hold the total; n * dan_deflate_bound(slot_bytes) bytes always do. Asynchronous on `stream`, so that a single
 * cudaMemcpyAsync of offsets[n] bytes carries only the compressed bytes to the host. */
int dan_deflate_compact(const void* slots, const uint32_t* lengths, int n, uint64_t slot_bytes, void* dst, uint64_t* offsets, void* stream);

/* BGZF compression on the device, with dan_deflate_device's kernel in gzip framing. src[0, bytes) is cut as bgzip cuts it: into
 * n = ceil(bytes / DAN_BGZF_MAX_INPUT) pieces of DAN_BGZF_MAX_INPUT bytes, the last one shorter. Piece i becomes one complete BGZF block
 * in dst + i * DAN_BGZF_MAX_BLOCK: the 18-byte gzip header (1f 8b 08 04, MTIME 0, XFL 0, OS ff, XLEN 6, subfield 'B' 'C' with SLEN 2 and
 * BSIZE = block size - 1), raw DEFLATE (dynamic-Huffman blocks, or one stored block when that is smaller; at most 18 + 5 + 65280 + 8 =
 * 65311 bytes in all), then the CRC-32 and ISIZE of the piece, all little-endian. block_lengths[i] receives the block's size and
 * status[i] DAN_DEFLATE_OK. The CRC-32 is computed in chunks and combined in a fixed order, so a block's bytes depend only on its
 * piece: not on the other pieces, the launch or the device. All pointers are DEVICE pointers (dst: n * DAN_BGZF_MAX_BLOCK bytes,
 * block_lengths and status: n entries); asynchronous on `stream`. bytes = 0 makes no blocks and launches nothing; otherwise a null
 * pointer returns DAN_E_INVALID before any launch. The 28-byte empty EOF block that ends a BGZF file is the caller's to append. */
#define DAN_BGZF_MAX_INPUT 65280
#define DAN_BGZF_MAX_BLOCK 65536
int dan_bgzf_compress_device(const void* src, uint64_t bytes, void* dst, uint32_t* block_lengths, int32_t* status, void* stream);

/* Packs the n blocks of dan_bgzf_compress_device back to back, as dan_deflate_compact does with slots DAN_BGZF_MAX_BLOCK apart:
 * offsets (DEVICE, n + 1 u64) receives the exclusive prefix sum of lengths and block i moves to dst + offsets[i]. */
int dan_bgzf_compact(const void* slots, const uint32_t* lengths, int n, void* dst, uint64_t* offsets, void* stream);

/* ---- device decode, of raw (DAN_RECORDS_RAW) or compressed (DAN_RECORDS_ZLIB) records --------------------------------------------
 * The caller stages the n records of a call in one pinned HOST buffer, at the offsets dan_decode_layout reports. The regions come in
 * this order, each 16-byte aligned, at offsets that depend only on (format, n); a region the format does not use is empty:
 *   [sidecars][records][stream offsets][stream lengths][headers][ref masks][var masks][streams]
 *   RAW:  records  = n records back to back, DAN_RECORD_BYTES apart;
 *   ZLIB: sidecars = n sidecars, DAN_SIDECAR_BYTES apart; stream offsets / lengths = n u64 / n u32, an offset counting from the
 *         start of the streams region; streams = room for n streams of up to max_stream_bytes.
 *   both: headers = n dan_record_header, ref / var masks = n * 201 bytes each, written by the call's header pass.
 * staging_bytes and workspace_bytes are the sizes of the staging buffer and of the DEVICE workspace for n records (and, for ZLIB, n
 * streams of max_stream_bytes, so sizes taken for a capacity serve every call of up to that many records). DAN_E_INVALID for an
 * unknown format or n < 0. */
enum { DAN_RECORDS_RAW = 0, DAN_RECORDS_ZLIB = 1 };
typedef struct dan_staging_layout {
  size_t sidecars, records, stream_offsets, stream_lengths, headers, ref_masks, var_masks, streams;   /* staging offsets */
  size_t staging_bytes, workspace_bytes;
} dan_staging_layout;
int dan_decode_layout(int format, int n, size_t max_stream_bytes, dan_staging_layout* out);

/* Device decode. Record i of the staging buffer decodes into candidate i; indices[i] is its index in its file, which seeds the read
 * draw exactly as in dan_decode_records. The call runs the header pass on the host (over the records, or over the sidecars for ZLIB),
 * writing the headers and masks into the staging buffer and the scalars of `out` (HOST pointers: label .. status, each may be NULL,
 * valid on return). One cudaMemcpyAsync on `stream` moves everything from the records region to the end of the last stream into
 * `workspace` (DEVICE); for ZLIB, dan_inflate_device then inflates the streams into n record images in the workspace and writes each
 * record's status to inflate_status (DEVICE, n int32; NULL for RAW). The tile pass then writes out->reads / q_scores / strands / ref /
 * ref_masks / var_masks (DEVICE pointers; q_scores / strands may be NULL). Every output equals dan_decode_records' on the raw records
 * byte for byte; a record whose stream fails to inflate gets all-zero tiles, ref and masks.
 * Before any header pass, copy or launch: DAN_E_INVALID for bad arguments or config, DAN_E_WORKSPACE if the staging buffer is too
 * small, DAN_E_INVALID if an index entry leaves the streams region, DAN_E_WORKSPACE if the workspace is too small for the streams
 * actually staged. Records the reference's loader raises on return DAN_E_INVALID with per-record status, as dan_decode_records.
 * Asynchronous: neither buffer may be reused before the stream has passed this call. */
int dan_decode_records_device(int format, void* staging, size_t staging_bytes, const int64_t* indices, int n, const dan_feeder_config* cfg,
                              const dan_record_batch* out, void* workspace, size_t workspace_bytes, int32_t* inflate_status, void* stream);

/* Test hook for the bit-exact integer/encoding work (dl4vc/model.py:450-627,719): writes the conv-1 input in the
 * reference's logical order (batch, Cin, num_reads, read_len) fp32, DEVICE pointer. */
int dan_encode(dan_model* m, const uint8_t* reads, const uint8_t* q_scores, const uint8_t* strands,
               const uint8_t* ref, const uint8_t* ref_masks, const uint8_t* var_masks, int batch,
               float* x0_out, void* stream);

/* Same hook for the bf16 path: what the fused conv-stack kernel's encoder prologue builds in shared memory for every read (bf16
 * planes, 45 -> 48 channels), widened to fp32 in the same (batch, Cin, num_reads, read_len) order — bf16_rn of the reference values,
 * match masks exactly 0 / 1. DAN_E_UNSUPPORTED for channel sets other than the shipped one (those use the fp32 encoder's rows). */
int dan_encode_bf16(dan_model* m, const uint8_t* reads, const uint8_t* q_scores, const uint8_t* strands,
                    const uint8_t* ref, const uint8_t* ref_masks, const uint8_t* var_masks, int batch,
                    float* x0_out, void* stream);

/* Test hook: after a dan_forward call on `workspace`, copy the FC input vector (pooled max|mean, or relu(post_pool(pooled)) when
 * pool_combine_dimension > 0, then relu(highway); dl4vc/model.py:838-912) of the LAST internal pass to out (rows x fc_in_features fp32, DEVICE pointer).
 * Returns the number of rows written, or a negative error. */
int dan_debug_fc_input(dan_model* m, int precision, int batch, const void* workspace, float* out, void* stream);

/* Kernel launches issued by the last dan_forward on this thread (for the benchmark's gpu_launches claim). */
int dan_last_launch_count(void);

/* Measurement aid for bench.py: the fp32 FMA rate this GPU sustains (TFLOP/s, 2 FLOP per FFMA) — a register-resident FFMA loop on every SM for
 * about `ms` milliseconds, timed with CUDA events on `stream`. The fp32 parity path and the training kernels run on this pipe; bench.py reports
 * this sustained figure (a pure FFMA loop is power-limited: ~54 of the nominal 74 TFLOP/s on B200) beside the nominal peak. Returns a negative
 * value on a CUDA error. */
double dan_measure_fma_tflops(double ms, void* stream);

/* Measurement hook (bench.py roofline): when enabled, every kernel launch of dan_forward is bracketed by CUDA
 * events on the launching stream, grouped in DAN_PROF_* classes. dan_profile_enable(1) also clears earlier
 * spans. dan_profile_read waits for the recorded events and returns the number of spans; ms_by_class /
 * launches_by_class receive the summed device time and launch count per class. */
enum { DAN_PROF_CONV_STACK = 0, DAN_PROF_GEMM = 1, DAN_PROF_ENCODE = 2, DAN_PROF_POOL = 3, DAN_PROF_NUM_CLASSES = 4 };
int dan_profile_enable(int on);
int dan_profile_read(double* ms_by_class, int* launches_by_class, int num_classes);
const char* dan_profile_class_name(int cls);

#ifdef __cplusplus
}
#endif
#endif /* DAN_B200_H */
