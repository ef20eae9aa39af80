"""Host-side feeder and score post-processing around the DAN forward (SURVEY §8f rows 1-2; north_star item 4).

PinnedBatchFeeder  collates the loader's per-candidate dicts (the schema `dl4vc/dataset.py:672-680` yields: uint8 `reads`,
                   `q-scores`, `strands` of shape (201, 100), `ref`, `ref_mask`, `var_mask` of shape (201,)) straight into
                   rotating PINNED uint8 batch buffers — no int64 inflation (`trainer.py:520-528` moves 8x the bytes) — and
                   hands them to `Basic2DNet.forward_heads_host`, whose library side overlaps the H2D staging of a chunk
                   with the kernels of the previous one. Collating batch k+1 on the host overlaps the GPU work of batch k.
scores_from_heads  the caller-side post-ops of `trainer.py:611-623`: softmax over xbinary / xVT and the variant score 1 - p0.
make_mask_vectors  batch proposal-mask decode of the loader (`dataset.py:112-250`) in the C-ABI library, pinned to the reference's outputs.
scores_on_device   the same post-ops as one CUDA kernel behind the C-ABI (`dan_scores`): 4 floats per candidate leave the GPU.
RecordFile / decode_records  raw fixed-record pileup file (the reference's HDF5 compound type as a flat np.memmap: h5py is not in the image) and
                   the batched C decode of `ContextDatasetFromNumpy._get_generator` (`dataset.py:500-680`: row window, sample_single_reads,
                   parse_vcf, count_variants_from_single_reads, proposal masks) straight into a pinned HostBatch — no per-item Python.
decode_records_device  the same decode with the tile pass on the GPU (`dan_decode_records_device`): host header pass (parse, sampling,
                   masks), one H2D copy of the staged raw records, a kernel that writes the device tiles `dan_forward` reads.
CompressedRecordFile  the same records as one zlib stream each, with an index and per-record sidecars (the bytes the header pass
                   reads); write_compressed_records writes one, with host zlib or on the GPU (`dan_deflate_device`), and
                   decode_records_device inflates the records on the GPU (`dan_inflate_device`).
call_record_file   record file -> scored VCF lines and genotype calls, streamed in batches through a ring of pinned slots.
format_vcf_info    the `BP=..;NV=..;HV=..;OV=..` field `utils.append_vcf_records` splices into VCF column 3 (`utils.py:162-178`).
"""
from __future__ import annotations

import ctypes as C
import os
import zlib
from collections import deque

import numpy as np
import torch

ITEM_KEYS = (("reads", "reads"), ("q-scores", "q"), ("strands", "strands"), ("ref", "ref"), ("ref_mask", "ref_masks"),
             ("var_mask", "var_masks"))


class HostBatch:
    """One pinned (when CUDA is available) uint8 batch in the layout the C-ABI takes: [batch][position][read]."""

    def __init__(self, capacity: int, read_len: int = 201, num_reads: int = 100, pin: bool | None = None):
        pin = torch.cuda.is_available() if pin is None else pin
        mk = lambda *shape: (torch.empty(shape, dtype=torch.uint8).pin_memory() if pin else torch.empty(shape, dtype=torch.uint8))
        self.reads, self.q, self.strands = (mk(capacity, read_len, num_reads) for _ in range(3))
        self.ref, self.ref_masks, self.var_masks = (mk(capacity, read_len) for _ in range(3))
        self.capacity, self.size = capacity, 0
        self.meta = []

    def fill(self, items) -> "HostBatch":
        """Copy a list of dataset items into the buffers (values are 0..93, any integer dtype narrows losslessly)."""
        n = len(items)
        if n > self.capacity:
            raise ValueError(f"{n} items > capacity {self.capacity}")
        views = {"reads": self.reads.numpy(), "q": self.q.numpy(), "strands": self.strands.numpy(), "ref": self.ref.numpy(),
                 "ref_masks": self.ref_masks.numpy(), "var_masks": self.var_masks.numpy()}
        for i, it in enumerate(items):
            for key, dst in ITEM_KEYS:
                a = np.asarray(it[key])
                if a.shape != views[dst].shape[1:]:
                    raise ValueError(f"item {i}: '{key}' has shape {a.shape}, expected {views[dst].shape[1:]} (dataset.py:672-680)")
                views[dst][i] = a          # numpy casts to uint8
        self.size = n
        self.meta = [(it.get("name"), it.get("vcfrec")) for it in items]
        return self

    def tensors(self):
        n = self.size
        return self.reads[:n], self.ref[:n], self.q[:n], self.strands[:n], self.ref_masks[:n], self.var_masks[:n]


class PinnedBatchFeeder:
    """submit(items) -> pending result; results() yields (meta, heads[n, 27]) in submission order.

    `depth` host batches rotate: while the GPU works on batch k (asynchronously, on `stream`), batch k+1 is collated into the
    next pinned buffer. A buffer is reused only after its result has been consumed, so at most `depth` batches are in flight."""

    def __init__(self, model, batch_size: int, depth: int = 2, stream: torch.cuda.Stream | None = None):
        self.model, self.batch_size, self.depth = model, batch_size, depth
        self.stream = stream
        self.free = deque(HostBatch(batch_size, model.single_read_len, model.num_single_reads) for _ in range(depth))
        self.pending = deque()

    def submit(self, items):
        if not self.free:
            raise RuntimeError("all host batches are in flight: consume results() first")
        hb = self.free.popleft().fill(items)
        ctx = torch.cuda.stream(self.stream) if self.stream is not None else _null()
        with ctx:
            out = self.model.forward_heads_host(*hb.tensors())
            ev = torch.cuda.Event()
            ev.record()
        self.pending.append((hb, out, ev))

    def results(self, drain: bool = True):
        """Yield finished (meta, heads) pairs; with drain=True waits for everything submitted so far."""
        while self.pending and (drain or self.pending[0][2].query()):
            hb, out, ev = self.pending.popleft()
            ev.synchronize()
            heads = out[: hb.size].clone()
            meta = hb.meta
            self.free.append(hb)
            yield meta, heads


class _null:
    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False


def scores_from_heads(heads: torch.Tensor):
    """(B,27) head matrix -> (bin_score (B,), vt_probs (B,3)) exactly as trainer.test computes them (trainer.py:611-623,
    use_var_type_threshold off): bin_score = 1 - softmax(xbinary)[:,0]; vt_probs = softmax(xVT) = P{no variant, het, hom}."""
    xbinary, xvt = heads[:, 0:2], heads[:, 2:5]
    bin_score = 1.0 - torch.softmax(xbinary, dim=1)[:, 0]
    return bin_score, torch.softmax(xvt, dim=1)


def scores_on_device(heads: torch.Tensor) -> torch.Tensor:
    """Device version of `scores_from_heads` through the C-ABI (`dan_scores`, include/dan_b200.h): (B,27) CUDA head matrix ->
    (B,4) CUDA tensor [bin_score, P(no variant), P(het), P(hom)], so only 16 bytes per candidate cross PCIe on the way to
    the VCF writer. No CPU path: raises on a CPU tensor."""
    from . import _lib
    if not heads.is_cuda:
        raise RuntimeError("scores_on_device needs the CUDA head matrix written by forward_heads (no CPU path)")
    if heads.dim() != 2 or heads.shape[1] != 27 or heads.dtype != torch.float32:
        raise RuntimeError("heads must be (B, 27) float32")
    heads = heads.contiguous()
    out = torch.empty((heads.shape[0], 4), dtype=torch.float32, device=heads.device)
    with torch.cuda.device(heads.device):
        _lib.check(_lib.load_library().dan_scores(heads.data_ptr(), heads.shape[0], out.data_ptr(),
                                                   torch.cuda.current_stream().cuda_stream), "dan_scores")
    return out


CALL_THRESHOLD_FIELDS = ("snp", "snp_zygo", "indel", "indel_zygo", "long_indel", "long_indel_zygo", "delete", "delete_zygo")


def resolve_call_thresholds(snp=0.3, snp_zygo=0.5, indel=0.0, indel_zygo=0.5, long_indel=0.0, long_indel_zygo=0.5, delete=0.0, delete_zygo=0.5):
    """The threshold fall-backs of tools/format_vcf.py:57-80 (arguments = its command-line options, same defaults). The script leaves the
    delete pair unassigned when --indel_threshold is not given (and raises on the first short delete); here it follows the indel pair."""
    if not indel > 0.0:
        indel, indel_zygo = snp, snp_zygo
        long_indel, long_indel_zygo = indel, indel_zygo
        delete, delete_zygo = indel, indel_zygo
    else:
        if not long_indel > 0.0:
            long_indel, long_indel_zygo = indel, indel_zygo
        if not delete > 0.0:
            delete, delete_zygo = indel, indel_zygo
    return (snp, snp_zygo, indel, indel_zygo, long_indel, long_indel_zygo, delete, delete_zygo)


def genotype_calls(scores, ref_len, var_len, **thresholds):
    """Host restatement of the per-record part of tools/format_vcf.py:107-138, vectorised: (gt, q) with gt 0 = dropped, 1 = "0/1", 2 = "1/1"
    and q the script's quality bucket (-1 when dropped). `scores` (n, 4) = [BP, NV, HV, OV] as written into the VCF ("%.8f")."""
    t = resolve_call_thresholds(**thresholds)
    s = np.asarray(scores, dtype=np.float32)
    nv = np.rint(s[:, 1].astype(np.float64) * 1e8) / 1e8
    ov = np.rint(s[:, 3].astype(np.float64) * 1e8) / 1e8
    rl, vl = np.asarray(ref_len), np.asarray(var_len)
    snp, lng, dele = (rl == 1) & (vl == 1), (rl >= 3) | (vl >= 3), (rl > 1) & (vl == 1)
    thr = np.where(snp, t[0], np.where(lng, t[4], np.where(dele, t[6], t[2])))
    hz = np.where(snp, t[1], np.where(lng, t[5], np.where(dele, t[7], t[3])))
    margin = (1.0 - nv) - thr
    keep = margin >= 0.0
    gt = np.where(keep, np.where(ov >= hz, 2, 1), 0).astype(np.int8)
    q = np.where(keep, (margin / (1.0 - thr) * 50.0).astype(np.int64), -1).astype(np.int32)
    return gt, q


def genotype_calls_on_device(scores: torch.Tensor, ref_len: torch.Tensor, var_len: torch.Tensor, **thresholds):
    """Device version through the C-ABI (`dan_genotype_calls`): scores (B,4) CUDA float32 from `scores_on_device`, allele lengths (B,) int32
    CUDA tensors -> (gt int8, q int32) CUDA tensors. No CPU path."""
    import ctypes as C
    from . import _lib
    if not scores.is_cuda:
        raise RuntimeError("genotype_calls_on_device needs CUDA tensors (no CPU path; genotype_calls is the host restatement)")
    B = scores.shape[0]
    scores = scores.contiguous().float()
    rl = ref_len.to(device=scores.device, dtype=torch.int32).contiguous(); vl = var_len.to(device=scores.device, dtype=torch.int32).contiguous()
    gt = torch.empty(B, dtype=torch.int8, device=scores.device); q = torch.empty(B, dtype=torch.int32, device=scores.device)
    d = dict(zip(CALL_THRESHOLD_FIELDS, (0.3, 0.5, 0.0, 0.5, 0.0, 0.5, 0.0, 0.5)))
    d.update(thresholds)
    thr = (C.c_double * 8)(*[d[k] for k in CALL_THRESHOLD_FIELDS])
    with torch.cuda.device(scores.device):
        _lib.check(_lib.load_library().dan_genotype_calls(scores.data_ptr(), rl.data_ptr(), vl.data_ptr(), B, C.cast(thr, C.c_void_p), gt.data_ptr(), q.data_ptr(),
                                                           torch.cuda.current_stream().cuda_stream), "dan_genotype_calls")
    return gt, q


def format_vcf_info(bin_score, vt_probs):
    """The strings utils.append_vcf_records writes into VCF column 3 (utils.py:171-176), vectorised over the batch."""
    b = np.asarray(bin_score, dtype=np.float64)
    v = np.asarray(vt_probs, dtype=np.float64)
    return ["BP=%.8f;NV=%.8f;HV=%.8f;OV=%.8f" % (b[i], v[i, 0], v[i, 1], v[i, 2]) for i in range(len(b))]


def make_mask_vectors(ref_alleles, var_alleles, references, strict: bool = True):
    """Batch version of the loader's `get_read_mask_vectors` (dl4vc/dataset.py:112-250) through the C-ABI (`dan_make_mask_vectors`):
    REF / ALT strings of n VCF records + their encoded reference windows (n, 201) uint8 -> (ref_masks, var_masks, status), each mask
    (n, 201) uint8. `status[i]` != 0 marks a record the reference itself would have raised on (masks all zero); with `strict` those
    raise a RuntimeError like the reference's assert would."""
    import ctypes as C
    from . import _lib
    refs = np.ascontiguousarray(np.asarray(references, dtype=np.uint8))
    n = len(ref_alleles)
    if refs.shape != (n, 201) or len(var_alleles) != n:
        raise RuntimeError("references must be (n, 201) uint8 with one REF / ALT string per row")
    xs = (C.c_char_p * max(n, 1))(*[str(a).encode("ascii") for a in ref_alleles])
    ys = (C.c_char_p * max(n, 1))(*[str(a).encode("ascii") for a in var_alleles])
    rm = np.zeros((n, 201), np.uint8); vm = np.zeros((n, 201), np.uint8); st = np.zeros(n, np.int32)
    lib = _lib.load_library()
    rc = lib.dan_make_mask_vectors(xs, ys, refs.ctypes.data, n, rm.ctypes.data, vm.ctypes.data, st.ctypes.data)
    if rc != 0 and (strict or not st.any()):
        _lib.check(rc, "dan_make_mask_vectors")
    return rm, vm, st


def format_vcf_info_native(scores) -> list:
    """Same strings as `format_vcf_info` from a (B,4) float32 score matrix [bin_score, P(no variant), P(het), P(hom)] (the output of
    `scores_on_device`, copied to the host), formatted by the C-ABI's `dan_format_vcf_info` instead of a Python loop."""
    import ctypes as C
    from . import _lib
    arr = np.ascontiguousarray(np.asarray(scores, dtype=np.float32))
    if arr.ndim != 2 or arr.shape[1] != 4:
        raise RuntimeError("scores must be (B, 4)")
    n, stride = arr.shape[0], 56
    buf = C.create_string_buffer(max(n, 1) * stride)
    _lib.check(_lib.load_library().dan_format_vcf_info(arr.ctypes.data, n, C.addressof(buf), len(buf)), "dan_format_vcf_info")
    raw = buf.raw
    return [raw[i * stride:i * stride + 55].decode("ascii") for i in range(n)]


def splice_vcf_records(vcf_records, bin_score, vt_probs):
    """Records with the score field spliced in, one per line, as append_vcf_records would append them (utils.py:166-178)."""
    return _splice_info(vcf_records, format_vcf_info(bin_score, vt_probs))


def _splice_info(vcf_records, info):
    if len(info) != len(vcf_records):
        raise AssertionError("mis-match between results and VCF to save")          # utils.py:165
    out = []
    for rec, txt in zip(vcf_records, info):
        items = rec.strip().split("\t")
        assert items[2] == ".", "DANGER -- would replace non-empty INFO -- check the hack"   # utils.py:172
        items[2] = txt
        out.append("\t".join(items))
    return out


# ---- raw record files + batched decode (dan_decode_records) --------------------------------------------------------------------------
RECORD_DTYPE = np.dtype([("name", "S16"), ("ref", np.uint8, (5, 201)), ("reads", np.uint16, (5, 201)), ("single_reads", np.uint8, (200, 201)),
                         ("ref_bases", np.uint8, (201,)), ("num_reads", np.int32), ("label", np.uint8), ("vcfrec", "S128"),
                         ("q-scores", np.uint8, (200, 201)), ("strand", np.uint8, (200, 201))])      # tools/convert_bam_single_reads.py:694-698
RECORD_BYTES = 123965
assert RECORD_DTYPE.itemsize == RECORD_BYTES
REC_STATUS = {0: "ok", 1: "vcf record has too few columns", 2: "allele letter outside base_enum", 3: "unknown mutation (equal-length non-SNP)",
              4: "INFO column without AF= / DP=", 5: "proposal masks: the reference raises (not an assertion)",
              6: "compressed record is corrupt"}
REC_CORRUPT = 6
# dan_inflate_device's per-stream status (DAN_INFLATE_*)
INFLATE_STATUS = {0: "ok", 1: "bad zlib header", 2: "bad block type", 3: "bad code set", 4: "distance too far back", 5: "input exhausted",
                  6: "output longer than its slot", 7: "output shorter than its slot", 8: "Adler-32 mismatch"}


class RecordFile:
    """np.memmap over back-to-back records of RECORD_DTYPE (what `hdfile['data']` holds in the reference, dataset.py:501-503)."""

    def __init__(self, path_or_array):
        if isinstance(path_or_array, np.ndarray):
            a = path_or_array
            self.raw = np.ascontiguousarray(a.view(np.uint8).reshape(len(a), -1)) if a.dtype == RECORD_DTYPE else np.ascontiguousarray(a, dtype=np.uint8)
        else:
            self.raw = np.memmap(path_or_array, dtype=np.uint8, mode="r").reshape(-1, RECORD_BYTES)
        assert self.raw.ndim == 2 and self.raw.shape[1] == RECORD_BYTES

    def __len__(self):
        return self.raw.shape[0]

    def field(self, idx, name):
        return self.raw[idx].view(RECORD_DTYPE)[0][name]

    def read_block(self, start: int, count: int, out):
        """Copy records [start, start + count) into the first count * RECORD_BYTES bytes of `out` (a uint8 numpy array or CPU tensor,
        typically pinned staging) with one memcpy; nothing is decoded."""
        if start < 0 or count < 0 or start + count > len(self):
            raise IndexError(f"records [{start}, {start + count}) outside the file's {len(self)}")
        dst = _byte_view(out, count)
        np.copyto(dst, self.raw[start:start + count].reshape(-1))

    def gather(self, indices, out):
        """Copy the records `indices` (any order, repeats allowed) back to back into `out`, like read_block does for a range."""
        idx = np.ascontiguousarray(np.asarray(indices, dtype=np.int64))
        if len(idx) and (idx.min() < 0 or idx.max() >= len(self)):
            raise IndexError("record index out of range")
        dst = _byte_view(out, len(idx))
        np.take(self.raw, idx, axis=0, out=dst.reshape(len(idx), RECORD_BYTES))


def _byte_view(out, count):
    a = out.numpy() if isinstance(out, torch.Tensor) else out
    if a.dtype != np.uint8 or a.ndim != 1 or not a.flags.c_contiguous:
        raise ValueError("out must be a contiguous 1-D uint8 buffer")
    if a.size < count * RECORD_BYTES:
        raise ValueError(f"out holds {a.size} bytes, {count} records need {count * RECORD_BYTES}")
    return a[:count * RECORD_BYTES]


# ---- compressed record files (layout: include/dan_b200.h) ----------------------------------------------------------------------------
COMPRESSED_MAGIC = b"DL4VCZR1"
SIDECAR_BYTES = 750
_CZ_HEADER = np.dtype([("magic", "S8"), ("version", "<u4"), ("record_bytes", "<u4"), ("count", "<u8"), ("index_off", "<u8"),
                       ("sidecar_off", "<u8"), ("data_off", "<u8"), ("data_bytes", "<u8"), ("sidecar_bytes", "<u4"), ("reserved", "<u4")])
_CZ_INDEX = np.dtype([("offset", "<u8"), ("length", "<u4")])
assert _CZ_HEADER.itemsize == 64 and _CZ_INDEX.itemsize == 12
# the sidecar as dan_record_sidecars cuts it (include/dan_b200.h); col100 / col101: single_reads columns 100 / 101 of the 200 stored rows
SIDECAR_DTYPE = np.dtype([("name", "S16"), ("num_reads", "<i4"), ("label", "u1"), ("vcfrec", "S128"), ("ref_bases", "u1", (201,)),
                          ("col100", "u1", (200,)), ("col101", "u1", (200,))])
assert SIDECAR_DTYPE.itemsize == SIDECAR_BYTES


def record_sidecars(raw) -> np.ndarray:
    """(n, RECORD_BYTES) uint8 records -> (n, SIDECAR_BYTES) sidecars, cut by the library (`dan_record_sidecars`), which alone knows
    which bytes the header pass reads."""
    from . import _lib
    raw = np.ascontiguousarray(raw)
    out = np.empty((len(raw), SIDECAR_BYTES), np.uint8)
    _lib.check(_lib.load_library().dan_record_sidecars(raw.ctypes.data, RECORD_BYTES, len(raw), out.ctypes.data), "dan_record_sidecars")
    return out


def _raw_rows(a) -> np.ndarray:
    a = np.asarray(a)
    if a.dtype == RECORD_DTYPE:
        return np.ascontiguousarray(a).reshape(-1).view(np.uint8).reshape(-1, RECORD_BYTES)
    if a.dtype == np.uint8 and a.ndim == 2 and a.shape[1] == RECORD_BYTES:
        return np.ascontiguousarray(a)
    raise ValueError(f"records must be RECORD_DTYPE or (n, {RECORD_BYTES}) uint8, not {a.dtype} {a.shape}")


def _source_chunks(source, chunk=256):
    if isinstance(source, RecordFile):
        for lo in range(0, len(source), chunk):
            yield source.raw[lo:lo + chunk]
    elif isinstance(source, np.ndarray):
        raw = _raw_rows(source)
        for lo in range(0, len(raw), chunk):
            yield raw[lo:lo + chunk]
    else:
        for a in source:
            yield _raw_rows(a)


def write_compressed_records(path, source, level: int | None = None, threads: int | None = None, device=None) -> int:
    """Write records as a compressed record file: one zlib stream per record. `source` is a RecordFile, a RECORD_DTYPE array, or an
    iterable of such arrays (e.g. slices of an HDF5 dataset), which is consumed once and never held whole. Returns the number of
    records written.

    device=None: standard-library zlib at `level` (default 6) on a pool of `threads` threads (zlib releases the GIL).
    device=<CUDA device>: the records are compressed on that GPU (`dan_deflate_device`, see deflate_device); `level` and `threads`
    do not apply and raise ValueError when given. The file's layout is the same either way; the streams differ, and both inflate to
    the records."""
    path = os.fspath(path)
    if device is None:
        chunks = _host_deflate_chunks(source, 6 if level is None else level, threads)
    else:
        dev = torch.device(device)
        if dev.type != "cuda":
            raise ValueError(f"device must be a CUDA device, not {dev}")
        if level is not None or threads is not None:
            raise ValueError("level and threads apply to host compression (device=None); the GPU deflate has one setting")
        chunks = _device_deflate_chunks(source, dev)
    return _write_compressed(path, chunks)


def _write_compressed(path, chunks) -> int:
    """The file around the streams: `chunks` yields (stream bytes back to back, their lengths, the chunk's sidecars)."""
    import contextlib
    import shutil
    import tempfile
    index, count, data_bytes = [], 0, 0
    pad = lambda f, k: f.write(b"\0" * (-k % 16)) and None
    with contextlib.closing(chunks), open(path, "wb") as f, tempfile.TemporaryFile(dir=os.path.dirname(os.path.abspath(path))) as side:
        f.write(b"\0" * 64)
        for data, lens, sidecars in chunks:
            lens = np.asarray(lens, dtype=np.uint64)
            entry = np.empty(len(lens), _CZ_INDEX)
            entry["offset"] = data_bytes + np.concatenate(([0], np.cumsum(lens)[:-1])).astype(np.uint64) if len(lens) else []
            entry["length"] = lens
            index.append(entry)
            f.write(data)
            side.write(sidecars.tobytes())
            data_bytes += int(lens.sum())
            count += len(lens)
        pad(f, data_bytes)
        sidecar_off = 64 + data_bytes + (-data_bytes % 16)
        side.seek(0)
        shutil.copyfileobj(side, f)
        pad(f, count * SIDECAR_BYTES)
        index_off = sidecar_off + count * SIDECAR_BYTES + (-(count * SIDECAR_BYTES) % 16)
        f.write((np.concatenate(index) if index else np.zeros(0, _CZ_INDEX)).tobytes())
        h = np.zeros(1, _CZ_HEADER)
        h[0] = (COMPRESSED_MAGIC, 1, RECORD_BYTES, count, index_off, sidecar_off, 64, data_bytes, SIDECAR_BYTES, 0)
        f.seek(0)
        f.write(h.tobytes())
    return count


def _host_deflate_chunks(source, level, threads):
    from concurrent.futures import ThreadPoolExecutor
    with ThreadPoolExecutor(threads or min(32, os.cpu_count() or 1)) as pool:
        for raw in _source_chunks(source):
            streams = list(pool.map(lambda r: zlib.compress(r.data, level), raw))
            yield b"".join(streams), [len(z) for z in streams], record_sidecars(raw)


class _DeflateSlot:
    """One chunk in flight on the GPU: pinned staging of the raw records, the device input, stream slots and packed output, and
    pinned landing buffers for the lengths / status and the packed streams."""

    def __init__(self, capacity, dev):
        bound = deflate_bound(RECORD_BYTES)
        self.capacity = capacity
        self.host_in = torch.empty(capacity * RECORD_BYTES, dtype=torch.uint8, pin_memory=True)
        self.dev_in = torch.empty(capacity * RECORD_BYTES, dtype=torch.uint8, device=dev)
        self.slots = torch.empty(capacity * bound, dtype=torch.uint8, device=dev)
        self.packed = torch.empty(capacity * bound, dtype=torch.uint8, device=dev)
        self.meta = torch.empty(2 * capacity, dtype=torch.int32, device=dev)            # lengths, then status
        self.offsets = torch.empty(capacity + 1, dtype=torch.int64, device=dev)
        self.host_meta = torch.empty(2 * capacity, dtype=torch.int32, pin_memory=True)
        self.host_out = torch.empty(capacity * bound, dtype=torch.uint8, pin_memory=True)
        self.done = torch.cuda.Event()
        self.job = None                                                                   # (first record, count, sidecars)


def _device_deflate_chunks(source, dev, depth=2):
    """GPU compression of _source_chunks(source). Per chunk: the records into a pinned slot, one H2D copy, dan_deflate_device,
    dan_deflate_compact, one D2H copy of lengths and status; once those have landed, one D2H copy of exactly the compressed bytes.
    `depth` slots rotate, so reading chunk k + 1 and cutting its sidecars on the host overlap the GPU work of chunk k."""
    from . import _lib
    lib = _lib.load_library()
    stream, copy_stream = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    slots, first = [], 0

    def finish(slot):
        start, n, sidecars = slot.job
        slot.job = None
        slot.done.synchronize()
        lens, status = slot.host_meta[:n].numpy().view(np.uint32).copy(), slot.host_meta[slot.capacity:slot.capacity + n].numpy()
        bad = np.flatnonzero(status != 0)
        if len(bad):
            raise RuntimeError(f"record #{start + int(bad[0])}: GPU deflate failed with status {int(status[bad[0]])}")
        total = int(lens.sum(dtype=np.uint64))
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(slot.done)
            slot.host_out[:total].copy_(slot.packed[:total], non_blocking=True)
        copy_stream.synchronize()
        return memoryview(slot.host_out[:total].numpy()), lens, sidecars

    try:
        with torch.cuda.device(dev):
            stream.wait_stream(torch.cuda.current_stream(dev))
            for k, raw in enumerate(_source_chunks(source)):
                n = len(raw)
                if len(slots) < depth:
                    slots.append(None)
                slot = slots[k % depth]
                if slot is not None and slot.job is not None:
                    yield finish(slot)
                if slot is None or slot.capacity < n:
                    slot = slots[k % depth] = _DeflateSlot(max(n, 1), dev)
                    stream.wait_stream(torch.cuda.current_stream(dev))
                if n:
                    np.copyto(slot.host_in[:n * RECORD_BYTES].numpy(), raw.reshape(-1))
                with torch.cuda.stream(stream):
                    slot.dev_in[:n * RECORD_BYTES].copy_(slot.host_in[:n * RECORD_BYTES], non_blocking=True)
                    st = stream.cuda_stream
                    _lib.check(lib.dan_deflate_device(slot.dev_in.data_ptr(), n, RECORD_BYTES, slot.slots.data_ptr(), slot.meta.data_ptr(),
                                                      slot.meta.data_ptr() + 4 * slot.capacity, st), "dan_deflate_device")
                    _lib.check(lib.dan_deflate_compact(slot.slots.data_ptr(), slot.meta.data_ptr(), n, RECORD_BYTES, slot.packed.data_ptr(),
                                                       slot.offsets.data_ptr(), st), "dan_deflate_compact")
                    slot.host_meta.copy_(slot.meta, non_blocking=True)
                    slot.done.record(stream)
                slot.job = (first, n, record_sidecars(raw))
                first += n
            pending = sorted((s for s in slots if s is not None and s.job is not None), key=lambda s: s.job[0])
            for slot in pending:
                yield finish(slot)
    finally:
        stream.synchronize()
        copy_stream.synchronize()


class CompressedRecordFile:
    """A compressed record file (write_compressed_records). Opening it checks the header and every index entry against the file's
    size and raises ValueError on a malformed file, before any record is read. The header pass runs on the sidecars; the records
    themselves are inflated on the GPU by decode_records_device, or on the host by `records`."""

    def __init__(self, path):
        self.path = os.fspath(path)
        size = os.path.getsize(self.path)
        if size < 64:
            raise ValueError(f"{self.path}: {size} bytes, shorter than the 64-byte header of a compressed record file")
        mm = np.memmap(self.path, dtype=np.uint8, mode="r")
        h = mm[:64].view(_CZ_HEADER)[0]
        if bytes(h["magic"]) != COMPRESSED_MAGIC:
            raise ValueError(f"{self.path}: not a compressed record file (magic {bytes(h['magic'])!r})")
        if int(h["version"]) != 1 or int(h["record_bytes"]) != RECORD_BYTES or int(h["sidecar_bytes"]) != SIDECAR_BYTES:
            raise ValueError(f"{self.path}: version {int(h['version'])}, {int(h['record_bytes'])}-byte records, {int(h['sidecar_bytes'])}-byte "
                             f"sidecars; this reader takes version 1, {RECORD_BYTES} and {SIDECAR_BYTES}")
        n = int(h["count"])
        for name, off, nbytes in (("index", int(h["index_off"]), n * _CZ_INDEX.itemsize), ("sidecar", int(h["sidecar_off"]), n * SIDECAR_BYTES),
                                  ("data", int(h["data_off"]), int(h["data_bytes"]))):
            if off < 64 or off > size or nbytes > size - off:
                raise ValueError(f"{self.path}: {name} section [{off}, +{nbytes}) lies outside the file's {size} bytes (truncated?)")
        ix = int(h["index_off"])
        index = np.frombuffer(mm[ix:ix + n * _CZ_INDEX.itemsize].tobytes(), _CZ_INDEX)
        self.offsets, self.lengths = index["offset"].astype(np.uint64), index["length"].astype(np.uint32)
        db = np.uint64(h["data_bytes"])
        bad = np.flatnonzero((self.offsets > db) | (self.lengths.astype(np.uint64) > db - np.minimum(self.offsets, db)))
        if len(bad):
            raise ValueError(f"{self.path}: index entry of record {int(bad[0])} points past the data section's end ({len(bad)} such entries)")
        so, do = int(h["sidecar_off"]), int(h["data_off"])
        self.sidecars = mm[so:so + n * SIDECAR_BYTES].reshape(n, SIDECAR_BYTES)
        self.data = mm[do:do + int(db)]
        self.max_stream_bytes = int(self.lengths.max()) if n else 0

    def __len__(self):
        return len(self.offsets)

    def stream(self, i) -> memoryview:
        o = int(self.offsets[i])
        return memoryview(self.data[o:o + int(self.lengths[i])])

    def field(self, idx, name):
        if name in ("name", "num_reads", "label", "vcfrec", "ref_bases"):
            return self.sidecars[idx].view(SIDECAR_DTYPE)[0][name]
        return self.records([idx])[0][name]

    def records(self, indices) -> np.ndarray:
        """Host inflate of `indices` (standard-library zlib) -> RECORD_DTYPE array. ValueError on a corrupt record."""
        idx = _record_indices(self, indices)
        out = np.empty(len(idx), RECORD_DTYPE)
        raw = out.view(np.uint8).reshape(len(idx), RECORD_BYTES)
        for k, i in enumerate(idx):
            try:
                rec = zlib.decompress(self.stream(int(i)))
            except zlib.error as e:
                raise ValueError(f"record {int(i)}: {e}") from None
            if len(rec) != RECORD_BYTES:
                raise ValueError(f"record {int(i)} inflates to {len(rec)} bytes, not {RECORD_BYTES}")
            raw[k] = np.frombuffer(rec, np.uint8)
        return out

    def unpack(self, path, chunk: int = 256):
        """Write the records back as a raw record file (RecordFile's format)."""
        with open(os.fspath(path), "wb") as f:
            for lo in range(0, len(self), chunk):
                f.write(self.records(np.arange(lo, min(len(self), lo + chunk))).tobytes())


def open_record_file(path):
    """A RecordFile, or a CompressedRecordFile when the file starts with the compressed magic."""
    with open(os.fspath(path), "rb") as f:
        head = f.read(len(COMPRESSED_MAGIC))
    return CompressedRecordFile(path) if head == COMPRESSED_MAGIC else RecordFile(os.fspath(path))


def inflate_device(src: torch.Tensor, offsets: torch.Tensor, lengths: torch.Tensor, slot_bytes: int, stream=None):
    """Inflate n zlib streams on the GPU (`dan_inflate_device`): stream i is src[offsets[i] : offsets[i] + lengths[i]] of the CUDA uint8
    tensor `src`; -> (dst (n, slot_bytes) uint8, status (n,) int32), CUDA tensors. status[i] == 0 (INFLATE_STATUS) means stream i
    inflated to exactly slot_bytes and passed its Adler-32 check; a failed stream leaves an all-zero row."""
    from . import _lib
    if not src.is_cuda or src.dtype != torch.uint8 or src.dim() != 1:
        raise ValueError("src must be a 1-D CUDA uint8 tensor")
    off = offsets.to(device=src.device, dtype=torch.int64).contiguous()
    ln = lengths.to(device=src.device, dtype=torch.int32).contiguous()
    n = off.numel()
    if ln.numel() != n:
        raise ValueError("one length per offset")
    o, l = off.cpu().numpy(), ln.cpu().numpy()
    if n and (o.min() < 0 or l.min() < 0 or (o + l).max() > src.numel()):
        raise ValueError("a stream lies outside src")
    dst = torch.empty((n, slot_bytes), dtype=torch.uint8, device=src.device)
    status = torch.empty(n, dtype=torch.int32, device=src.device)
    with torch.cuda.device(src.device):
        st = (stream if stream is not None else torch.cuda.current_stream(src.device)).cuda_stream
        _lib.check(_lib.load_library().dan_inflate_device(src.data_ptr(), off.data_ptr(), ln.data_ptr(), n, dst.data_ptr(), slot_bytes, status.data_ptr(), st),
                   "dan_inflate_device")
    return dst, status


def deflate_bound(slot_bytes: int) -> int:
    """Bytes of one output slot of dan_deflate_device: the stored-block encoding of slot_bytes, which no stream exceeds."""
    from . import _lib
    return int(_lib.load_library().dan_deflate_bound(slot_bytes))


def deflate_device(src: torch.Tensor, stream=None):
    """Compress the n rows of the CUDA uint8 tensor `src` (n, slot) on the GPU (`dan_deflate_device`), each into one standard zlib
    stream that zlib.decompress and inflate_device both take; the mirror of inflate_device. -> (streams, offsets, lengths, status),
    CUDA tensors: the streams packed back to back in one uint8 tensor, stream i at streams[offsets[i] : offsets[i] + lengths[i]]
    (int64 / int32), and status[i] == 0 (DAN_DEFLATE_OK) for each. Waits for the device to learn the packed size."""
    from . import _lib
    if not isinstance(src, torch.Tensor) or not src.is_cuda or src.dtype != torch.uint8 or src.dim() != 2:
        raise ValueError("src must be a 2-D (n, slot) CUDA uint8 tensor")
    src = src.contiguous()
    n, slot = src.shape
    lib = _lib.load_library()
    bound = int(lib.dan_deflate_bound(slot))
    dev = src.device
    slots = torch.empty(n * bound, dtype=torch.uint8, device=dev)
    packed = torch.empty(n * bound, dtype=torch.uint8, device=dev)
    lengths = torch.empty(n, dtype=torch.int32, device=dev)
    status = torch.empty(n, dtype=torch.int32, device=dev)
    offsets = torch.empty(n + 1, dtype=torch.int64, device=dev)
    with torch.cuda.device(dev):
        stream = stream if stream is not None else torch.cuda.current_stream(dev)
        st = stream.cuda_stream
        _lib.check(lib.dan_deflate_device(src.data_ptr(), n, slot, slots.data_ptr(), lengths.data_ptr(), status.data_ptr(), st),
                   "dan_deflate_device")
        _lib.check(lib.dan_deflate_compact(slots.data_ptr(), lengths.data_ptr(), n, slot, packed.data_ptr(), offsets.data_ptr(), st),
                   "dan_deflate_compact")
        stream.synchronize()
        total = int(offsets[n].item())
    return packed[:total], offsets[:n], lengths, status


_SCALARS = (("label", np.uint8), ("num_reads", np.int32), ("is_snp", np.uint8), ("var_type", np.int32), ("allele_freq", np.float32),
            ("coverage", np.int32), ("var_base_enum", np.int32), ("var_ref_enum", np.int32), ("blacklist", np.uint8), ("status", np.int32))


# dan_record_header (include/dan_b200.h): tile column j < num_rows of every tile is stored row rows[j]
RECORD_HEADER_DTYPE = np.dtype([("window_start", np.int32), ("num_rows", np.int32), ("ref_len", np.int32), ("var_len", np.int32),
                                ("rows", np.uint8, (200,))])
assert RECORD_HEADER_DTYPE.itemsize == 216


def _feeder_cfg(max_reads, store_max_reads, use_q_scores, use_strands, keep_candidate_af, seed):
    from . import _lib
    return _lib.DanFeederConfigC(max_reads, store_max_reads, int(use_q_scores), int(use_strands), int(keep_candidate_af), int(seed))


def _record_indices(records, indices):
    idx = np.ascontiguousarray(np.asarray(indices, dtype=np.int64)).reshape(-1)
    if len(idx) and (idx.min() < 0 or idx.max() >= len(records)):
        raise IndexError(f"record index out of range [0, {len(records)})")
    return idx


def _scalars(n):
    return {k: np.zeros(n, t) for k, t in _SCALARS}


def _batch_struct(tiles, sc):
    from . import _lib
    ptr = lambda t: None if t is None else t.data_ptr() if isinstance(t, torch.Tensor) else t.ctypes.data
    return _lib.DanRecordBatchC(*[ptr(t) for t in tiles], *[sc[k].ctypes.data for k, _ in _SCALARS])


def _raise_failed(idx, sc):
    bad = np.flatnonzero(sc["status"])
    raise ValueError(f"{len(bad)} records cannot be decoded (the reference loader raises on them): " +
                     ", ".join(f"#{int(idx[b])}: {REC_STATUS.get(int(sc['status'][b]), '?')}" for b in bad[:5]))


def decode_records(records: RecordFile, indices, batch: HostBatch | None = None, use_q_scores=True, use_strands=True, keep_candidate_af=False, seed=0,
                   max_reads=100, store_max_reads=200, strict=True):
    """Decode `indices` of a RecordFile into a (pinned) HostBatch + the per-example scalars the trainer reads (dataset.py:672-680).
    Returns (batch, scalars dict of numpy arrays incl. `status` / `blacklist`). strict: raise if the reference's loader would."""
    from . import _lib
    lib = _lib.load_library()
    idx = _record_indices(records, indices)
    n = len(idx)
    if batch is None:
        batch = HostBatch(max(n, 1), num_reads=max_reads)
    if n > batch.capacity:
        raise ValueError(f"{n} records > capacity {batch.capacity}")
    sc = _scalars(n)
    out = _batch_struct((batch.reads, batch.q, batch.strands, batch.ref, batch.ref_masks, batch.var_masks), sc)
    cfg = _feeder_cfg(max_reads, store_max_reads, use_q_scores, use_strands, keep_candidate_af, seed)
    rc = lib.dan_decode_records(records.raw.ctypes.data, RECORD_BYTES, idx.ctypes.data, n, C.byref(cfg), C.byref(out))
    batch.size = n
    batch.meta = [(bytes(records.field(int(i), "name")).decode(), bytes(records.field(int(i), "vcfrec")).decode()) for i in idx]
    if rc < 0 and strict:
        _raise_failed(idx, sc)
    return batch, sc


def decode_record_headers(records, indices, use_q_scores=True, use_strands=True, keep_candidate_af=False, seed=0, max_reads=100,
                          store_max_reads=200):
    """The header pass of the decode alone (`dan_decode_record_headers`, host code): -> (headers, scalars, ref_masks, var_masks).
    headers is a RECORD_HEADER_DTYPE array; scalars and masks are what decode_records returns for the same arguments. On a
    CompressedRecordFile the pass runs over the sidecars (`dan_decode_sidecar_headers`) with the same results."""
    from . import _lib
    lib = _lib.load_library()
    idx = _record_indices(records, indices)
    n = len(idx)
    sc = _scalars(n)
    rm, vm = np.zeros((n, 201), np.uint8), np.zeros((n, 201), np.uint8)
    hdr = np.zeros(n, RECORD_HEADER_DTYPE)
    out = _batch_struct((None, None, None, None, rm, vm), sc)
    cfg = _feeder_cfg(max_reads, store_max_reads, use_q_scores, use_strands, keep_candidate_af, seed)
    if isinstance(records, CompressedRecordFile):
        rc = lib.dan_decode_sidecar_headers(records.sidecars.ctypes.data, idx.ctypes.data, n, C.byref(cfg), C.byref(out), hdr.ctypes.data)
    else:
        rc = lib.dan_decode_record_headers(records.raw.ctypes.data, RECORD_BYTES, idx.ctypes.data, n, C.byref(cfg), C.byref(out), hdr.ctypes.data)
    if rc < 0 and not sc["status"].any():
        _lib.check(rc, "dan_decode_record_headers")
    return hdr, sc, rm, vm


def _decode_layout(fmt, n, max_stream_bytes=0):
    """The staging layout of n records of format fmt (_lib.RECORDS_RAW / RECORDS_ZLIB), as dan_decode_layout reports it."""
    from . import _lib
    lay = _lib.DanStagingLayoutC()
    _lib.check(_lib.load_library().dan_decode_layout(fmt, n, max_stream_bytes, C.byref(lay)), "dan_decode_layout")
    return lay


class DeviceBatch:
    """Decoded batch on the GPU (`dan_decode_records_device`): device uint8 tiles in the layout dan_forward takes, the pinned host
    staging buffer the records are read into, and the device workspace they are copied to. The decoded tiles exist only on the
    device.

    With `max_stream_bytes` (a CompressedRecordFile's largest stream) the batch decodes compressed records: the staging buffer holds
    sidecars and zlib streams, sized for `capacity` streams of that size, and `inflate_status` is a device int32 tensor with each
    record's inflate status (INFLATE_STATUS) of the last decode."""

    def __init__(self, capacity: int, num_reads: int = 100, device=None, read_len: int = 201, max_stream_bytes: int | None = None):
        from . import _lib
        if not 1 <= num_reads <= 200:
            raise ValueError(f"max_reads {num_reads} out of range 1..200")
        dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.capacity, self.num_reads, self.device, self.size = capacity, num_reads, dev, 0
        self.max_stream_bytes = max_stream_bytes
        self.format = _lib.RECORDS_RAW if max_stream_bytes is None else _lib.RECORDS_ZLIB
        lay = _decode_layout(self.format, capacity, max_stream_bytes or 0)
        self.inflate_status = None if max_stream_bytes is None else torch.zeros(capacity, dtype=torch.int32, device=dev)
        self.staging = torch.empty(lay.staging_bytes, dtype=torch.uint8).pin_memory()
        self.workspace = torch.empty(lay.workspace_bytes, dtype=torch.uint8, device=dev)
        mk = lambda *shape: torch.empty(shape, dtype=torch.uint8, device=dev)
        self.reads, self.q, self.strands = (mk(capacity, read_len, num_reads) for _ in range(3))
        self.ref, self.ref_masks, self.var_masks = (mk(capacity, read_len) for _ in range(3))
        self.meta = []

    def tensors(self):
        n = self.size
        return self.reads[:n], self.ref[:n], self.q[:n], self.strands[:n], self.ref_masks[:n], self.var_masks[:n]

    def headers(self):
        """Header-pass descriptors of the last decode (RECORD_HEADER_DTYPE, a view into the staging buffer)."""
        n = self.size
        off = _decode_layout(self.format, n).headers
        return self.staging.numpy()[off:off + n * RECORD_HEADER_DTYPE.itemsize].view(RECORD_HEADER_DTYPE)


def decode_records_device(records, indices, batch: DeviceBatch | None = None, use_q_scores=True, use_strands=True,
                          keep_candidate_af=False, seed=0, max_reads=100, store_max_reads=200, strict=True, stream=None):
    """decode_records with the tile pass on the GPU (`dan_decode_records_device`). The records go into the batch's pinned staging
    buffer (one memcpy from the file for a contiguous ascending range, an index gather otherwise), the header pass runs on the host,
    then one H2D copy and the tile kernel run on `stream` (default: the current stream). Returns (batch, scalars) with the same
    outputs as decode_records, byte for byte. Asynchronous: the batch's tensors are ready once `stream` has passed the call, and
    the batch may be decoded into again only after that.

    `records` is a RecordFile, a CompressedRecordFile or a path (opened by its magic). For a compressed file the zlib streams are
    staged instead of the records, the header pass runs over the sidecars, and the records are inflated on the GPU before the tile
    pass; the batch must be a compressed DeviceBatch (default: one sized for the file). The call does not wait for the inflate:
    `batch.inflate_status` holds each record's status once `stream` has passed the call, and a record whose stream is corrupt
    decodes to all-zero tiles and masks."""
    from . import _lib
    if not isinstance(records, (RecordFile, CompressedRecordFile)):
        records = open_record_file(records)
    compressed = isinstance(records, CompressedRecordFile)
    idx = _record_indices(records, indices)
    n = len(idx)
    if batch is None:
        batch = DeviceBatch(max(n, 1), num_reads=max_reads, max_stream_bytes=records.max_stream_bytes if compressed else None)
    if n > batch.capacity:
        raise ValueError(f"{n} records > capacity {batch.capacity}")
    if batch.num_reads != max_reads:
        raise ValueError(f"batch holds {batch.num_reads} reads per candidate, max_reads is {max_reads}")
    if compressed != (batch.max_stream_bytes is not None):
        raise ValueError("a compressed record file needs a DeviceBatch with max_stream_bytes, a raw one a DeviceBatch without")
    lay = _decode_layout(batch.format, n)
    st = batch.staging.numpy()
    if compressed:
        st[lay.sidecars:lay.sidecars + n * SIDECAR_BYTES].reshape(n, SIDECAR_BYTES)[:] = records.sidecars[idx]
        st[lay.stream_offsets:lay.stream_offsets + 8 * n].view(np.uint64)[:] = _stage_streams(records, idx, st[lay.streams:])
        st[lay.stream_lengths:lay.stream_lengths + 4 * n].view(np.uint32)[:] = records.lengths[idx]
        rows = st[lay.sidecars:lay.sidecars + n * SIDECAR_BYTES].view(SIDECAR_DTYPE)
    else:
        if n and np.all(np.diff(idx) == 1):
            records.read_block(int(idx[0]), n, st[lay.records:])
        else:
            records.gather(idx, st[lay.records:])
        rows = st[lay.records:lay.records + n * RECORD_BYTES].view(RECORD_DTYPE)
    sc = _scalars(n)
    out = _batch_struct((batch.reads, batch.q, batch.strands, batch.ref, batch.ref_masks, batch.var_masks), sc)
    cfg = _feeder_cfg(max_reads, store_max_reads, use_q_scores, use_strands, keep_candidate_af, seed)
    with torch.cuda.device(batch.device):
        s = (stream if stream is not None else torch.cuda.current_stream(batch.device)).cuda_stream
        rc = _lib.load_library().dan_decode_records_device(batch.format, batch.staging.data_ptr(), batch.staging.numel(), idx.ctypes.data, n,
                                                           C.byref(cfg), C.byref(out), batch.workspace.data_ptr(), batch.workspace.numel(),
                                                           None if batch.inflate_status is None else batch.inflate_status.data_ptr(), s)
    batch.size = n
    batch.meta = [(a.decode(), b.decode()) for a, b in zip(rows["name"].tolist(), rows["vcfrec"].tolist())]
    if rc == -1 and sc["status"].any():          # DAN_E_INVALID with per-record status: records the reference raises on
        if strict:
            _raise_failed(idx, sc)
    else:
        _lib.check(rc, "dan_decode_records_device")
    return batch, sc


def _stage_streams(rf: CompressedRecordFile, idx, dst: np.ndarray):
    """Copy the streams of records idx back to back into dst; -> their offsets in dst. A contiguous ascending range whose streams
    lie back to back in the file (as write_compressed_records lays them out) is one copy."""
    n = len(idx)
    off, ln = rf.offsets[idx], rf.lengths[idx].astype(np.uint64)
    if n and np.all(np.diff(idx) == 1) and np.all(off[1:] == off[:-1] + ln[:-1]):
        span = int(off[-1] + ln[-1] - off[0])
        if span > dst.size:
            raise ValueError(f"{n} streams of {span} bytes exceed the batch's {dst.size}-byte stream region")
        dst[:span] = rf.data[int(off[0]):int(off[0]) + span]
        return off - off[0]
    pos = np.concatenate(([0], np.cumsum(ln))).astype(np.uint64)
    if n and int(pos[-1]) > dst.size:
        raise ValueError(f"{n} streams of {int(pos[-1])} bytes exceed the batch's {dst.size}-byte stream region")
    for k, i in enumerate(idx):
        o = int(rf.offsets[i])
        dst[int(pos[k]):int(pos[k + 1])] = rf.data[o:o + int(rf.lengths[i])]
    return pos[:n]


class _CallSlot:
    """One ring slot of call_record_file: a DeviceBatch plus the pinned buffers of its allele lengths and results."""

    def __init__(self, capacity, num_reads, dev, max_stream_bytes=None):
        self.batch = DeviceBatch(capacity, num_reads, dev, max_stream_bytes=max_stream_bytes)
        pin = lambda shape, dt: torch.empty(shape, dtype=dt).pin_memory()
        self.ref_len, self.var_len = pin(capacity, torch.int32), pin(capacity, torch.int32)
        self.scores, self.gt, self.q = pin((capacity, 4), torch.float32), pin(capacity, torch.int8), pin(capacity, torch.int32)
        self.inflate_status = None if max_stream_bytes is None else pin(capacity, torch.int32)


def call_record_file(model, records, start=0, stop=None, batch_size=1036, depth=2, thresholds=None, strict=True, failed=None, seed=0,
                     store_max_reads=200, keep_candidate_af=False):
    """Stream records [start, stop) of a record file (a path, opened by its magic, a RecordFile or a CompressedRecordFile) to scored VCF
    records and genotype calls: the whole path of
    the reference's inference (main.py --test_file -> trainer.test -> append_vcf_records -> tools/format_vcf.py's thresholds) in one call.

    Yields, per batch of up to `batch_size` records in file order, (names, vcf_lines, gt, q): record names, the VCF records with the
    score field spliced in (exactly what splice_vcf_records writes), and the genotype calls of genotype_calls_on_device (gt int8 numpy:
    0 dropped, 1 "0/1", 2 "1/1"; q int32 numpy). `thresholds` are genotype_calls' keyword arguments.

    Per batch: the records are read into a pinned ring slot (one memcpy), the header pass runs on the host, and the H2D copy and the
    device tile pass run on a side stream; forward_heads, dan_scores and dan_genotype_calls follow on the current stream, and only
    scores (16 bytes) and gt / q per record come back. `depth` slots rotate, so the host work of batch k+1 overlaps the GPU work of
    batch k; a slot is reused only after its batch's results have been yielded.
    Records the reference's loader raises on (status != 0): strict=True raises naming them; strict=False leaves them out and appends
    (record index, status) to `failed` when a list is given.
    From a compressed file the streams are staged and inflated on the device; a record whose stream is corrupt gets status
    REC_CORRUPT and is handled the same way. Its inflate status is known only once the batch's device work has finished, so a strict
    raise for it comes when that batch is finished (after the batches before it have been yielded), not when it is submitted."""
    rf = records if isinstance(records, (RecordFile, CompressedRecordFile)) else open_record_file(records)
    msb = rf.max_stream_bytes if isinstance(rf, CompressedRecordFile) else None
    stop = len(rf) if stop is None else int(stop)
    start = int(start)
    if not 0 <= start <= stop <= len(rf):
        raise IndexError(f"record range [{start}, {stop}) outside the file's {len(rf)}")
    if batch_size < 1 or depth < 1:
        raise ValueError("batch_size and depth must be >= 1")
    if model.training:
        raise RuntimeError("call_record_file runs the eval-mode forward: call .eval() first")
    dev = model._device()
    thr = dict(thresholds or {})
    opts = dict(use_q_scores=model.use_q_scores, use_strands=model.use_strands, keep_candidate_af=keep_candidate_af, seed=seed,
                max_reads=model.num_single_reads, store_max_reads=store_max_reads)
    with torch.cuda.device(dev):
        main, side = torch.cuda.current_stream(dev), torch.cuda.Stream(dev)
        free = deque(_CallSlot(min(batch_size, max(stop - start, 1)), model.num_single_reads, dev, msb) for _ in range(depth))
        side.wait_stream(main)          # the slots' device memory may be blocks the current stream freed with work still queued on them
        pending = deque()

        def submit(b0, n):
            slot = free.popleft()
            idx = np.arange(b0, b0 + n, dtype=np.int64)
            batch, sc = decode_records_device(rf, idx, slot.batch, strict=False, stream=side, **opts)
            bad = np.flatnonzero(sc["status"])
            if strict and len(bad):
                side.synchronize()      # the copy and tile pass just queued still use the slot
                free.append(slot)
                _raise_failed(idx, sc)
            hdr = batch.headers()
            slot.ref_len[:n].numpy()[:] = hdr["ref_len"]
            slot.var_len[:n].numpy()[:] = hdr["var_len"]
            main.wait_stream(side)
            with torch.cuda.stream(main):
                heads = model.forward_heads(*batch.tensors())
                scores = scores_on_device(heads)
                rl, vl = slot.ref_len[:n].to(dev, non_blocking=True), slot.var_len[:n].to(dev, non_blocking=True)
                gt, q = genotype_calls_on_device(scores, rl, vl, **thr)
                slot.scores[:n].copy_(scores, non_blocking=True)
                slot.gt[:n].copy_(gt, non_blocking=True)
                slot.q[:n].copy_(q, non_blocking=True)
                if slot.inflate_status is not None:
                    slot.inflate_status[:n].copy_(batch.inflate_status[:n], non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(main)
            pending.append((slot, idx, sc["status"].copy(), batch.meta, ev))

        def finish():
            slot, idx, status, meta, ev = pending.popleft()
            ev.synchronize()
            n = len(idx)
            if slot.inflate_status is not None:
                status = np.where((status == 0) & (slot.inflate_status[:n].numpy() != 0), REC_CORRUPT, status)
                if strict and (status == REC_CORRUPT).any():
                    free.append(slot)
                    _raise_failed(idx, {"status": status})
            good = status == 0
            if failed is not None:
                failed.extend((int(idx[b]), int(status[b])) for b in np.flatnonzero(~good))
            keep = np.flatnonzero(good)
            scores = slot.scores[:n].numpy()[keep]
            names = [meta[k][0] for k in keep]
            lines = _splice_info([meta[k][1] for k in keep], format_vcf_info_native(scores))
            out = (names, lines, slot.gt[:n].numpy()[keep].copy(), slot.q[:n].numpy()[keep].copy())
            free.append(slot)
            return out

        try:
            for b0 in range(start, stop, batch_size):
                if not free:
                    yield finish()
                submit(b0, min(batch_size, stop - b0))
            while pending:
                yield finish()
        finally:
            # on an exception or an abandoned generator the slots are freed here: let the device work that uses them finish first
            # (the raw staging copies are invisible to torch's allocators)
            side.synchronize()
            for *_, ev in pending:
                ev.synchronize()
