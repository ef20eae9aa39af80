// dan_feeder.cu — batched decode of pileup records into the model-facing uint8 tensors (SURVEY §8f-1). Host code.
//
// Replaces the per-item Python path of the reference loader, ContextDatasetFromNumpy._get_generator (dl4vc/dataset.py:500-680) with its
// helpers sample_single_reads (:256-287), parse_vcf (dl4vc/utils.py:19-72), count_variants_from_single_reads (:340-362) and
// get_read_mask_vectors (:112-250), for a whole batch of record indices at once, writing straight into (pinned) host buffers in the
// layout dan_forward_host takes: [candidate][position][read]. Records are the compound type tools/convert_bam_single_reads.py writes
// (:694-698, SURVEY App. C) stored back to back as raw bytes (np.memmap of that dtype; h5py / libhdf5 are not in this image).
#include <cstdlib>
#include <string>
#include "dan_records.h"

namespace {

// field offsets of the packed record (numpy compound dtype without alignment), --max-reads 200 --window-size 100
constexpr int kRecP = DAN_MASK_READ_LEN;      // 201 columns
constexpr int kRecRows = 200;                 // stored read rows (TOTAL_SINGLE_READS)
constexpr size_t kOffName = 0, kOffRef5 = 16, kOffReads5 = kOffRef5 + 5 * kRecP, kOffSingle = kOffReads5 + 2 * 5 * kRecP,
                 kOffRefBases = kOffSingle + (size_t)kRecRows * kRecP, kOffNumReads = kOffRefBases + kRecP, kOffLabel = kOffNumReads + 4,
                 kOffVcf = kOffLabel + 1, kOffQ = kOffVcf + 128, kOffStrand = kOffQ + (size_t)kRecRows * kRecP, kRecBytes = kOffStrand + (size_t)kRecRows * kRecP;
static_assert(kRecBytes == DAN_RECORD_BYTES, "record layout");

inline uint64_t splitmix(uint64_t& x) {
  x += 0x9E3779B97F4A7C15ull;
  uint64_t z = x;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull; z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}

struct VcfInfo { int is_snp, var_mode, ref_base, var_base, var_type, coverage; double allele_freq; };

// dl4vc/utils.py:19-72. Returns a DAN_REC_E_* status; every failure is one the reference raises on (KeyError / ValueError / IndexError).
int parse_vcf_record(const std::string& rec_in, VcfInfo* out, std::string* ref_allele, std::string* var_allele) {
  // str.strip() + split('\t')
  size_t b = 0, e = rec_in.size();
  while (b < e && isspace((unsigned char)rec_in[b])) ++b;
  while (e > b && isspace((unsigned char)rec_in[e - 1])) --e;
  std::vector<std::string> f;
  for (size_t i = b, start = b; i <= e; ++i)
    if (i == e || rec_in[i] == '\t') { f.emplace_back(rec_in.substr(start, i - start)); start = i + 1; }
  if (f.size() < 8) return DAN_REC_E_VCF_FIELDS;
  const std::string &x = f[3], &y = f[4];
  *ref_allele = x; *var_allele = y;
  VcfInfo r{};
  if (x.size() == 1 && y.size() == 1 && mask_real_base(x[0]) && mask_real_base(y[0])) {
    r.is_snp = 1; r.var_mode = 1;
    r.ref_base = mask_base_code(x[0]); r.var_base = mask_base_code(y[0]);
  } else if (x.size() > y.size()) {
    r.var_mode = 3;                                   // delete: GAAA -> G, reference base 'G', variant base '-'
    r.ref_base = mask_base_code(x[0]); r.var_base = 5;
  } else if (x.size() < y.size()) {
    if (x.empty()) return DAN_REC_E_ALLELE;           // ref_bases[0] raises IndexError
    r.var_mode = 2;                                   // insert: G -> GAAAA, variant base 'noinsert'
    r.ref_base = mask_base_code(x[0]); r.var_base = 8;
  } else {
    return DAN_REC_E_UNKNOWN_MUTATION;                // "Unknown mutation detected": no var_mode -> KeyError in the loader (dataset.py:596)
  }
  if (r.ref_base < 0 || r.var_base < 0) return DAN_REC_E_ALLELE;
  // INFO column: {n: v for (n, v) in [k.split('=') for k in rec[7].split(';')]}
  bool have_af = false, have_dp = false;
  const std::string& info = f[7];
  for (size_t i = 0, start = 0; i <= info.size(); ++i) {
    if (i != info.size() && info[i] != ';') continue;
    const std::string kv = info.substr(start, i - start);
    start = i + 1;
    const size_t eq = kv.find('=');
    if (eq == std::string::npos || kv.find('=', eq + 1) != std::string::npos) return DAN_REC_E_VCF_INFO;      // unpack of != 2 parts raises ValueError
    const std::string k = kv.substr(0, eq), v = kv.substr(eq + 1);
    if (k == "AF") {
      char* end = nullptr;
      r.allele_freq = strtod(v.c_str(), &end);
      if (end == v.c_str() || *end) return DAN_REC_E_VCF_INFO;
      have_af = true;
    } else if (k == "DP") {
      char* end = nullptr;
      const long dp = strtol(v.c_str(), &end, 10);
      if (end == v.c_str() || *end) return DAN_REC_E_VCF_INFO;
      r.coverage = (int)dp; have_dp = true;
    }
  }
  if (!have_af || !have_dp) return DAN_REC_E_VCF_INFO;
  r.var_type = 0;
  if (f.size() > 10) {
    const std::string& g = f[10];
    const size_t c = g.find(':');
    if (c == std::string::npos || g.find(':', c + 1) != std::string::npos) return DAN_REC_E_VCF_FIELDS;             // gt, var = rec[10].split(':')
    const std::string gt = g.substr(0, c), var = g.substr(c + 1);
    if (gt == "GT" && var.size() == 3 && (var[1] == '/' || var[1] == '|')) {
      if (var[0] == '1' && var[2] == '1') r.var_type = 2;
      else if ((var[0] == '0' && var[2] == '1') || (var[0] == '1' && var[2] == '0')) r.var_type = 1;
    }
  }
  *out = r;
  return DAN_REC_OK;
}

// ---- header pass: everything of the decode that is not tile bytes (host, shared by the host and the device decode) --------------
// Row window + sample_single_reads selection, parse_vcf, allele counts at the proposal column over the chosen rows, coverage /
// allele_freq, proposal masks, blacklist and status. Writes the scalars of record i into `out` (each may be NULL), the masks into
// rm / vm, and the chosen stored rows into *h. `key` seeds the draw of deep pileups (the record's index in its file).
// The pass reads its record through a HeaderView: the scalar fields, ref_bases, and single_reads columns 100 and 101 of the stored rows.

// sidecar layout (include/dan_b200.h): the bytes a HeaderView reads, plus the name
constexpr size_t kSideName = 0, kSideNumReads = 16, kSideLabel = 20, kSideVcf = 21, kSideRef = kSideVcf + 128, kSideCol100 = kSideRef + kRecP,
                 kSideCol101 = kSideCol100 + kRecRows, kSideBytes = kSideCol101 + kRecRows;
static_assert(kSideBytes == DAN_SIDECAR_BYTES, "sidecar layout");

struct HeaderView {
  const uint8_t *num_reads, *label, *vcf, *ref;
  const uint8_t* col[2];                      // single_reads columns 100 and 101: stored row r at col[c][r * row_stride]
  size_t row_stride;
};
HeaderView raw_view(const uint8_t* rec) {
  return {rec + kOffNumReads, rec + kOffLabel, rec + kOffVcf, rec + kOffRefBases, {rec + kOffSingle + 100, rec + kOffSingle + 101}, (size_t)kRecP};
}
HeaderView sidecar_view(const uint8_t* sc) {
  return {sc + kSideNumReads, sc + kSideLabel, sc + kSideVcf, sc + kSideRef, {sc + kSideCol100, sc + kSideCol101}, 1};
}

int header_pass(const HeaderView& rec, int64_t key, const dan_feeder_config* cfg, int R, int S, const dan_record_batch* out, int i,
                uint8_t* rm, uint8_t* vm, dan_record_header* h) {
  int32_t num_reads;
  memcpy(&num_reads, rec.num_reads, 4);
  // A. window of stored rows (dataset.py:517-521), B. at most R of them (sample_single_reads, dataset.py:256-287)
  const int middle = (num_reads > S ? num_reads : S) / 2;
  int start = (int)((double)middle - (double)S / 2.0);
  if (start < 0) start = 0;
  const int avail = start < kRecRows ? (kRecRows - start < S ? kRecRows - start : S) : 0;      // columns of the transposed window
  const int max_reads = R < avail ? R : avail;
  int perm[kRecRows];
  if (max_reads >= num_reads) {
    for (int j = 0; j < max_reads; ++j) perm[j] = j;                                              // the first max_reads columns, deterministic
  } else {
    // a sorted random subset of the first min(avail, num_reads) columns: the reference draws it with an unseeded np.random.choice
    // (its inference is not reproducible for deep pileups, SURVEY App. G); here the draw is a function of (seed, record index)
    const int total = avail < num_reads ? avail : num_reads;
    uint64_t st = cfg->seed ^ (0xD1B54A32D192ED03ull * (uint64_t)(key + 1));
    int pool[kRecRows];
    for (int j = 0; j < total; ++j) pool[j] = j;
    for (int j = 0; j < max_reads; ++j) { const int k = j + (int)(splitmix(st) % (uint64_t)(total - j)); const int t = pool[j]; pool[j] = pool[k]; pool[k] = t; }
    bool take[kRecRows] = {};
    for (int j = 0; j < max_reads; ++j) take[pool[j]] = true;
    for (int j = 0, k = 0; j < total; ++j) if (take[j]) perm[k++] = j;
  }
  memset(h, 0, sizeof(*h));
  h->window_start = start;
  h->num_rows = max_reads;
  for (int j = 0; j < max_reads; ++j) h->rows[j] = (uint8_t)(start + perm[j]);      // start + perm[j] < start + avail <= kRecRows
  const uint8_t* ref = rec.ref;
  if (out->label) out->label[i] = *rec.label;
  if (out->num_reads) out->num_reads[i] = num_reads;
  // vcfrec: S128, trailing NULs stripped like numpy does
  size_t len = 128;
  while (len > 0 && rec.vcf[len - 1] == 0) --len;
  const std::string vcf(reinterpret_cast<const char*>(rec.vcf), len);
  VcfInfo vi{};
  std::string xa, ya;
  int status = parse_vcf_record(vcf, &vi, &xa, &ya);
  h->ref_len = (int32_t)xa.size();
  h->var_len = (int32_t)ya.size();
  memset(rm, 0, kRecP); memset(vm, 0, kRecP);
  int blacklist = 0;
  if (status == DAN_REC_OK) {
    // coverage / allele frequency from the sampled reads at the proposal column (count_variants_from_single_reads, dataset.py:340-362);
    // tile column j of the reads holds stored row h->rows[j], so the column is read from the record itself
    int ref_base; int col;
    if (vi.var_mode == 1) { ref_base = ref[100]; col = 100; }
    else if (vi.var_mode == 3) { ref_base = ref[101]; col = 101; }
    else { ref_base = 8; col = 101; }
    int agree = 0, disagree = 0;
    for (int j = 0; j < max_reads; ++j) {
      const int t = rec.col[col - 100][(size_t)h->rows[j] * rec.row_stride];
      if (t == ref_base) ++agree;
      else if (t == 1 || t == 2 || t == 3 || t == 4 || t == 5 || t == 8 || t == 9) ++disagree;      // real_base_keys_set: A T C G - M noinsert
    }
    // columns beyond max_reads do not exist in the reference's slice: only the chosen rows count
    const int cover = agree + disagree;
    int coverage = vi.coverage; double af = vi.allele_freq;
    if (cover > 0) { coverage = cover; if (!cfg->keep_candidate_af) af = (double)disagree / (double)cover; }
    if (out->is_snp) out->is_snp[i] = (uint8_t)vi.is_snp;
    if (out->var_type) out->var_type[i] = vi.var_type;
    if (out->allele_freq) out->allele_freq[i] = (float)af;
    if (out->coverage) out->coverage[i] = coverage;
    if (out->var_base_enum) out->var_base_enum[i] = vi.var_base;
    if (out->var_ref_enum) out->var_ref_enum[i] = vi.ref_base;
    // proposal masks (get_read_mask_vectors); an AssertionError there blacklists the example and leaves all-pad masks (dataset.py:644-664)
    const int mcode = mask_one(xa.c_str(), ya.c_str(), ref, rm, vm);
    if (mcode != DAN_MASK_OK) {
      memset(rm, 0, kRecP); memset(vm, 0, kRecP);
      if (mcode == DAN_MASK_E_SHAPE || mcode == DAN_MASK_E_REF_MISMATCH) blacklist = 1;      // assert -> caught
      else status = DAN_REC_E_MASK;                                                            // KeyError / ValueError / UnboundLocalError propagate in the reference
    }
  }
  if (out->blacklist) out->blacklist[i] = (uint8_t)blacklist;
  if (out->status) out->status[i] = status;
  return status;
}

// host tile pass: tile column j = stored row h.rows[j] transposed to [position][read]; columns past num_rows stay zero
void host_tiles(const uint8_t* rec, const dan_record_header& h, const dan_feeder_config* cfg, int R, const dan_record_batch* out, int i) {
  const size_t tile = (size_t)kRecP * R;
  uint8_t* reads = out->reads + (size_t)i * tile;
  uint8_t* q = out->q_scores ? out->q_scores + (size_t)i * tile : nullptr;
  uint8_t* sd = out->strands ? out->strands + (size_t)i * tile : nullptr;
  memset(reads, 0, tile);
  if (q) memset(q, 0, tile);
  if (sd) memset(sd, 0, tile);
  for (int j = 0; j < h.num_rows; ++j) {
    const uint8_t* row = rec + kOffSingle + (size_t)h.rows[j] * kRecP;
    const uint8_t* qrow = rec + kOffQ + (size_t)h.rows[j] * kRecP;
    const uint8_t* srow = rec + kOffStrand + (size_t)h.rows[j] * kRecP;
    for (int p = 0; p < kRecP; ++p) {
      reads[(size_t)p * R + j] = row[p];
      if (q && cfg->use_q_scores) q[(size_t)p * R + j] = qrow[p];
      if (sd && cfg->use_strands) sd[(size_t)p * R + j] = srow[p];
    }
  }
  memcpy(out->ref + (size_t)i * kRecP, rec + kOffRefBases, kRecP);
}

// The checks every batch entry point starts with: the count, the pointers (`pointers` is false if one is NULL), the record stride
// and the config, whose read counts go to R / S. Nothing is checked past the count when n == 0.
int check_batch(int n, bool pointers, const dan_feeder_config* cfg, int* R, int* S, size_t record_stride = DAN_RECORD_BYTES) {
  if (n < 0) { dan_set_error("negative record count"); return DAN_E_INVALID; }
  if (n == 0) return DAN_OK;
  if (!pointers || !cfg) { dan_set_error("null pointer"); return DAN_E_INVALID; }
  if (record_stride < DAN_RECORD_BYTES) { dan_set_error("record stride %zu below the %d-byte record", record_stride, DAN_RECORD_BYTES); return DAN_E_INVALID; }
  *R = cfg->max_reads; *S = cfg->store_max_reads < kRecRows ? cfg->store_max_reads : kRecRows;
  if (*R < 1 || *R > kRecRows || *S < 1) { dan_set_error("max_reads %d / store_max_reads %d out of range", *R, cfg->store_max_reads); return DAN_E_INVALID; }
  return DAN_OK;
}

// The header pass over n records, record i read through view(i) and keyed by indices[i]; its masks go to rm / vm + i * 201 and its
// header to headers[i].
template <class View>
int header_passes(View view, const int64_t* indices, int n, const dan_feeder_config* cfg, int R, int S, const dan_record_batch* out,
                  uint8_t* rm, uint8_t* vm, dan_record_header* headers) {
  int failed = 0;
  for (int i = 0; i < n; ++i)
    if (header_pass(view(i), indices[i], cfg, R, S, out, i, rm + (size_t)i * kRecP, vm + (size_t)i * kRecP, headers + i) != DAN_REC_OK) ++failed;
  if (failed) { dan_set_error("%d of %d records raise in the reference loader (see status[])", failed, n); return DAN_E_INVALID; }
  return DAN_OK;
}

// ---- device tile pass ------------------------------------------------------------------------------------------------------------
constexpr size_t align16(size_t x) { return (x + 15) & ~(size_t)15; }

// The staging layout of include/dan_b200.h. The device workspace holds the n record images (for ZLIB; for RAW they are the copied
// records region) followed by the staging buffer from the records region on, so every copied region keeps its 16-byte alignment.
dan_staging_layout staging_layout(int format, int n, size_t max_stream_bytes) {
  const bool zlib = format == DAN_RECORDS_ZLIB;
  dan_staging_layout l;
  size_t at = 0;
  auto region = [&](size_t bytes) { const size_t o = at; at = align16(at + bytes); return o; };
  l.sidecars = region(zlib ? (size_t)n * kSideBytes : 0);
  l.records = region(zlib ? 0 : (size_t)n * kRecBytes);
  l.stream_offsets = region(zlib ? (size_t)n * 8 : 0);
  l.stream_lengths = region(zlib ? (size_t)n * 4 : 0);
  l.headers = region((size_t)n * sizeof(dan_record_header));
  l.ref_masks = region((size_t)n * kRecP);
  l.var_masks = region((size_t)n * kRecP);
  l.streams = at;
  l.staging_bytes = align16(l.streams + (zlib ? (size_t)n * max_stream_bytes : 0));
  l.workspace_bytes = (zlib ? align16((size_t)n * kRecBytes) : 0) + l.staging_bytes - l.records;
  return l;
}

constexpr int kTileThreads = 256;

// grid (n, 3): block (i, t) writes tile t (0 reads, 1 q-scores, 2 strands) of record i from its image images + i * DAN_RECORD_BYTES.
// The chosen rows are gathered into a [position][read] image of the tile in shared memory (zero past num_rows, or everywhere for a
// tile the config leaves unused), placed at the output address's offset mod 16, so the tile leaves shared memory in aligned 16-byte
// stores; only the bytes before the first and after the last 16-byte boundary of the record's range go out one by one. Blocks of
// tile 0 also copy ref_bases and the header pass's masks. A record whose inflate_status (NULL for raw records) is not DAN_INFLATE_OK
// decodes to nothing: no tile rows and all-zero masks (its image, ref_bases included, is already all zero).
__global__ void decode_tiles_kernel(const uint8_t* __restrict__ images, const dan_record_header* __restrict__ headers,
                                    const uint8_t* __restrict__ rm, const uint8_t* __restrict__ vm, const int32_t* __restrict__ inflate_status,
                                    int R, int use_q, int use_s, uint8_t* __restrict__ reads, uint8_t* __restrict__ q, uint8_t* __restrict__ sd,
                                    uint8_t* __restrict__ ref, uint8_t* __restrict__ ref_masks, uint8_t* __restrict__ var_masks) {
  extern __shared__ uint4 tile_smem[];
  __shared__ uint8_t rows[kRecRows];
  const int i = blockIdx.x, t = blockIdx.y, tid = threadIdx.x;
  uint8_t* dst_base = t == 0 ? reads : t == 1 ? q : sd;
  if (!dst_base) return;
  const int T = kRecP * R;
  uint8_t* dst = dst_base + (size_t)i * T;
  const int mis = (int)((uintptr_t)dst & 15);
  uint8_t* s = reinterpret_cast<uint8_t*>(tile_smem) + mis;
  const dan_record_header* h = headers + i;
  const bool ok = !inflate_status || inflate_status[i] == DAN_INFLATE_OK;
  const int num_rows = ok ? h->num_rows : 0;
  const bool fill = t == 0 || (t == 1 && use_q) || (t == 2 && use_s);
  for (int k = tid; k < (T + 31) / 16; k += kTileThreads) tile_smem[k] = make_uint4(0, 0, 0, 0);
  if (tid < num_rows) rows[tid] = h->rows[tid];
  __syncthreads();
  const uint8_t* rec = images + (size_t)i * kRecBytes;
  if (fill) {
    const uint8_t* src = rec + (t == 0 ? kOffSingle : t == 1 ? kOffQ : kOffStrand);
    for (int e = tid; e < num_rows * kRecP; e += kTileThreads) {        // consecutive threads read consecutive bytes of one stored row
      const int j = e / kRecP, p = e - j * kRecP;
      s[p * R + j] = src[rows[j] * kRecP + p];
    }
  }
  __syncthreads();
  const int head = min((16 - mis) & 15, T);
  const int chunks = (T - head) >> 4;
  for (int k = tid; k < head; k += kTileThreads) dst[k] = s[k];
  const uint4* s4 = reinterpret_cast<const uint4*>(s + head);
  uint4* d4 = reinterpret_cast<uint4*>(dst + head);
  for (int k = tid; k < chunks; k += kTileThreads) d4[k] = s4[k];
  for (int k = head + chunks * 16 + tid; k < T; k += kTileThreads) dst[k] = s[k];
  if (t == 0) {
    const size_t o = (size_t)i * kRecP;
    for (int k = tid; k < kRecP; k += kTileThreads) {
      ref[o + k] = rec[kOffRefBases + k];
      ref_masks[o + k] = ok ? rm[o + k] : 0;
      var_masks[o + k] = ok ? vm[o + k] : 0;
    }
  }
}

}  // namespace

extern "C" {

int dan_decode_records(const void* records, size_t record_stride, const int64_t* indices, int n, const dan_feeder_config* cfg, const dan_record_batch* out) {
  int R, S;
  const int rc = check_batch(n, records && indices && out && out->reads && out->ref && out->ref_masks && out->var_masks, cfg, &R, &S, record_stride);
  if (rc != DAN_OK || n == 0) return rc;
  const auto rec = [&](int i) { return static_cast<const uint8_t*>(records) + (size_t)indices[i] * record_stride; };
  std::vector<dan_record_header> h(n);
  const int failed = header_passes([&](int i) { return raw_view(rec(i)); }, indices, n, cfg, R, S, out, out->ref_masks, out->var_masks, h.data());
  for (int i = 0; i < n; ++i) host_tiles(rec(i), h[i], cfg, R, out, i);
  return failed;
}

int dan_decode_record_headers(const void* records, size_t record_stride, const int64_t* indices, int n, const dan_feeder_config* cfg,
                              const dan_record_batch* out, dan_record_header* headers) {
  int R, S;
  const int rc = check_batch(n, records && indices && out && out->ref_masks && out->var_masks && headers, cfg, &R, &S, record_stride);
  if (rc != DAN_OK || n == 0) return rc;
  return header_passes([&](int i) { return raw_view(static_cast<const uint8_t*>(records) + (size_t)indices[i] * record_stride); }, indices, n, cfg,
                       R, S, out, out->ref_masks, out->var_masks, headers);
}

int dan_record_sidecars(const void* records, size_t record_stride, int n, void* out) {
  if (n < 0) { dan_set_error("negative record count"); return DAN_E_INVALID; }
  if (n == 0) return DAN_OK;
  if (!records || !out) { dan_set_error("null pointer"); return DAN_E_INVALID; }
  if (record_stride < DAN_RECORD_BYTES) { dan_set_error("record stride %zu below the %d-byte record", record_stride, DAN_RECORD_BYTES); return DAN_E_INVALID; }
  for (int i = 0; i < n; ++i) {
    const uint8_t* rec = static_cast<const uint8_t*>(records) + (size_t)i * record_stride;
    uint8_t* sc = static_cast<uint8_t*>(out) + (size_t)i * kSideBytes;
    memcpy(sc + kSideName, rec + kOffName, 16);
    memcpy(sc + kSideNumReads, rec + kOffNumReads, 4);
    sc[kSideLabel] = rec[kOffLabel];
    memcpy(sc + kSideVcf, rec + kOffVcf, 128);
    memcpy(sc + kSideRef, rec + kOffRefBases, kRecP);
    for (int r = 0; r < kRecRows; ++r) {
      sc[kSideCol100 + r] = rec[kOffSingle + (size_t)r * kRecP + 100];
      sc[kSideCol101 + r] = rec[kOffSingle + (size_t)r * kRecP + 101];
    }
  }
  return DAN_OK;
}

int dan_decode_sidecar_headers(const void* sidecars, const int64_t* indices, int n, const dan_feeder_config* cfg, const dan_record_batch* out,
                               dan_record_header* headers) {
  int R, S;
  const int rc = check_batch(n, sidecars && indices && out && out->ref_masks && out->var_masks && headers, cfg, &R, &S);
  if (rc != DAN_OK || n == 0) return rc;
  return header_passes([&](int i) { return sidecar_view(static_cast<const uint8_t*>(sidecars) + (size_t)indices[i] * kSideBytes); }, indices, n,
                       cfg, R, S, out, out->ref_masks, out->var_masks, headers);
}

int dan_decode_layout(int format, int n, size_t max_stream_bytes, dan_staging_layout* out) {
  if (format != DAN_RECORDS_RAW && format != DAN_RECORDS_ZLIB) { dan_set_error("unknown record format %d", format); return DAN_E_INVALID; }
  if (n < 0) { dan_set_error("negative record count"); return DAN_E_INVALID; }
  if (!out) { dan_set_error("null pointer"); return DAN_E_INVALID; }
  *out = staging_layout(format, n, max_stream_bytes);
  return DAN_OK;
}

int dan_decode_records_device(int format, void* staging, size_t staging_bytes, const int64_t* indices, int n, const dan_feeder_config* cfg,
                              const dan_record_batch* out, void* workspace, size_t workspace_bytes, int32_t* inflate_status, void* stream) {
  if (format != DAN_RECORDS_RAW && format != DAN_RECORDS_ZLIB) { dan_set_error("unknown record format %d", format); return DAN_E_INVALID; }
  const bool zlib = format == DAN_RECORDS_ZLIB;
  int R, S;
  int rc = check_batch(n, staging && indices && out && out->reads && out->ref && out->ref_masks && out->var_masks && workspace && (!zlib || inflate_status),
                       cfg, &R, &S);
  if (rc != DAN_OK || n == 0) return rc;
  const dan_staging_layout l = staging_layout(format, n, 0);      // the streams region is what the caller's buffer has room for
  if (staging_bytes < l.staging_bytes) {
    dan_set_error("staging buffer of %zu bytes is below the %zu bytes %d records need", staging_bytes, l.staging_bytes, n); return DAN_E_WORKSPACE;
  }
  uint8_t* st = static_cast<uint8_t*>(staging);
  const uint64_t* off = reinterpret_cast<const uint64_t*>(st + l.stream_offsets);
  const uint32_t* len = reinterpret_cast<const uint32_t*>(st + l.stream_lengths);
  const size_t cap = staging_bytes - l.streams;
  size_t used = 0;                                                // bytes of the streams region the copy carries
  for (int i = 0; zlib && i < n; ++i) {
    if (off[i] > cap || len[i] > cap - off[i]) {
      dan_set_error("stream %d ([%llu, +%u)) leaves the %zu-byte streams region of the staging buffer", i, (unsigned long long)off[i], len[i], cap);
      return DAN_E_INVALID;
    }
    if (off[i] + len[i] > used) used = off[i] + len[i];
  }
  if (workspace_bytes < l.workspace_bytes + used) {
    dan_set_error("device workspace of %zu bytes is below the %zu bytes %d records need", workspace_bytes, l.workspace_bytes + used, n);
    return DAN_E_WORKSPACE;
  }
  dan_record_header* hdr = reinterpret_cast<dan_record_header*>(st + l.headers);
  const int failed = zlib ? header_passes([&](int i) { return sidecar_view(st + l.sidecars + (size_t)i * kSideBytes); }, indices, n, cfg, R, S, out,
                                          st + l.ref_masks, st + l.var_masks, hdr)
                          : header_passes([&](int i) { return raw_view(st + l.records + (size_t)i * kRecBytes); }, indices, n, cfg, R, S, out,
                                          st + l.ref_masks, st + l.var_masks, hdr);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  uint8_t* ws = static_cast<uint8_t*>(workspace);               // the record images
  uint8_t* dev = ws + (l.workspace_bytes - l.staging_bytes);    // the device copy of staging byte b (b >= l.records) is dev + b
  DAN_CUDA_TRY(cudaMemcpyAsync(dev + l.records, st + l.records, l.streams - l.records + used, cudaMemcpyHostToDevice, s));
  if (zlib) {
    rc = dan_inflate_launch(dev + l.streams, reinterpret_cast<const uint64_t*>(dev + l.stream_offsets),
                            reinterpret_cast<const uint32_t*>(dev + l.stream_lengths), n, ws, kRecBytes, inflate_status, s);
    if (rc != DAN_OK) return rc;
  }
  const int smem = ((kRecP * R + 31) / 16) * 16;
  decode_tiles_kernel<<<dim3(n, 3), kTileThreads, smem, s>>>(ws, reinterpret_cast<const dan_record_header*>(dev + l.headers), dev + l.ref_masks,
                                                             dev + l.var_masks, zlib ? inflate_status : nullptr, R, cfg->use_q_scores != 0,
                                                             cfg->use_strands != 0, out->reads, out->q_scores, out->strands, out->ref,
                                                             out->ref_masks, out->var_masks);
  DAN_CUDA_TRY(cudaGetLastError());
  return failed;
}

}  // extern "C"
