"""BGZF-compressed, tabix-indexed VCF output: the `.vcf.gz` + `.tbi` pair that ends the reference pipeline (`call_variants.sh`:
sort -> format_vcf.py -> bcftools norm -> bgzip -> tabix), written from the lines call_record_file yields.

bgzf_compress_device  text -> BGZF blocks on the GPU (`dan_bgzf_compress_device`, the deflate kernel of dan_deflate.cu in BGZF framing).
BgzfVcfWriter         header + record lines -> `.vcf.gz` and its `.tbi`; the text is cut into 65280-byte pieces as bgzip cuts it,
                      compressed on the GPU or with host zlib, and indexed on the host.
write_scored_vcf      call_record_file straight into a BgzfVcfWriter, optionally sorted.
concat_vcf_shards     per-rank files -> one file and index, copying the compressed blocks as they are.

The index follows the SAM/tabix specification (format 2, VCF); see build_tabix_index for the rules.
"""
from __future__ import annotations

import array
import gzip
import os
import re
import struct
import time
import zlib

import numpy as np
import torch

BGZF_MAX_INPUT = 65280          # DAN_BGZF_MAX_INPUT: input bytes of a full block, as bgzip cuts
BGZF_MAX_BLOCK = 65536          # DAN_BGZF_MAX_BLOCK: the largest block, and the slot stride of dan_bgzf_compress_device
BGZF_EOF = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")
TBI_MAX_POS = 1 << 29           # .tbi coordinates (0-based) stay below this; larger ones need a CSI index
_PSEUDO_BIN = 37450


# ---- BGZF blocks ------------------------------------------------------------------------------------------------------------------
def bgzf_block(raw_deflate: bytes, data: bytes) -> bytes:
    """One BGZF block around the raw DEFLATE of `data`: the 18-byte gzip header with the BC subfield, then CRC-32 and ISIZE."""
    size = 18 + len(raw_deflate) + 8
    if size > BGZF_MAX_BLOCK:
        raise ValueError(f"a {size}-byte block exceeds BGZF's {BGZF_MAX_BLOCK}")
    return (b"\x1f\x8b\x08\x04\0\0\0\0\0\xff\x06\0BC\x02\0" + struct.pack("<H", size - 1) + raw_deflate
            + struct.pack("<II", zlib.crc32(data), len(data)))


def host_bgzf_blocks(data, level: int = 6) -> list:
    """data cut into BGZF_MAX_INPUT-byte pieces, each compressed with host zlib at `level` into one block."""
    out = []
    for lo in range(0, len(data), BGZF_MAX_INPUT):
        piece = bytes(data[lo:lo + BGZF_MAX_INPUT])
        c = zlib.compressobj(level, zlib.DEFLATED, -15)
        out.append(bgzf_block(c.compress(piece) + c.flush(), piece))
    return out


def bgzf_compress_device(src: torch.Tensor, stream=None):
    """Compress the 1-D CUDA uint8 tensor `src` into BGZF blocks on the GPU (`dan_bgzf_compress_device`): piece i =
    src[i * 65280 : (i + 1) * 65280] (the last one shorter) becomes one complete block. -> (blocks, offsets, lengths, status), CUDA
    tensors: the blocks packed back to back in one uint8 tensor, block i at blocks[offsets[i] : offsets[i] + lengths[i]] (int64 /
    int32), and status[i] == 0 (DAN_DEFLATE_OK) for each. The mirror of feeder.deflate_device; waits for the device to learn the
    packed size."""
    from . import _lib
    if not isinstance(src, torch.Tensor) or not src.is_cuda or src.dtype != torch.uint8 or src.dim() != 1:
        raise ValueError("src must be a 1-D CUDA uint8 tensor")
    src = src.contiguous()
    nbytes = src.numel()
    n = -(-nbytes // BGZF_MAX_INPUT)
    lib = _lib.load_library()
    dev = src.device
    slots = torch.empty(n * BGZF_MAX_BLOCK, dtype=torch.uint8, device=dev)
    packed = torch.empty(n * BGZF_MAX_BLOCK, dtype=torch.uint8, device=dev)
    lengths = torch.empty(n, dtype=torch.int32, device=dev)
    status = torch.empty(n, dtype=torch.int32, device=dev)
    offsets = torch.empty(n + 1, dtype=torch.int64, device=dev)
    with torch.cuda.device(dev):
        stream = stream if stream is not None else torch.cuda.current_stream(dev)
        st = stream.cuda_stream
        _lib.check(lib.dan_bgzf_compress_device(src.data_ptr(), nbytes, slots.data_ptr(), lengths.data_ptr(), status.data_ptr(), st),
                   "dan_bgzf_compress_device")
        _lib.check(lib.dan_bgzf_compact(slots.data_ptr(), lengths.data_ptr(), n, packed.data_ptr(), offsets.data_ptr(), st), "dan_bgzf_compact")
        stream.synchronize()
        total = int(offsets[n].item())
    return packed[:total], offsets[:n], lengths, status


class _BgzfSlot:
    """One batch of pieces in flight on the GPU: pinned staging of the text, the device input, block slots and packed output, and
    pinned landing buffers for the lengths / status and the packed blocks."""

    def __init__(self, pieces, dev):
        self.pieces = pieces
        cap = pieces * BGZF_MAX_INPUT
        self.host_in = torch.empty(cap, dtype=torch.uint8, pin_memory=True)
        self.dev_in = torch.empty(cap, dtype=torch.uint8, device=dev)
        self.slots = torch.empty(pieces * BGZF_MAX_BLOCK, dtype=torch.uint8, device=dev)
        self.packed = torch.empty(pieces * BGZF_MAX_BLOCK, dtype=torch.uint8, device=dev)
        self.meta = torch.empty(2 * pieces, dtype=torch.int32, device=dev)             # lengths, then status
        self.offsets = torch.empty(pieces + 1, dtype=torch.int64, device=dev)
        self.host_meta = torch.empty(2 * pieces, dtype=torch.int32, pin_memory=True)
        self.host_out = torch.empty(pieces * BGZF_MAX_BLOCK, dtype=torch.uint8, pin_memory=True)
        self.done = torch.cuda.Event()
        self.n = None                                                                     # pieces of the batch in flight


class _DeviceBgzf:
    """Text -> BGZF blocks on one GPU with `depth` rotating slots of up to `pieces` pieces. submit() queues a batch and returns the
    blocks of the batch that used the slot before, if any, so the host's work on the next batch overlaps the GPU's on this one.
    Per batch: one H2D copy, dan_bgzf_compress_device, dan_bgzf_compact, one D2H copy of lengths and status; once those have landed,
    one D2H copy of exactly the compressed bytes."""

    def __init__(self, dev, pieces, depth=2):
        from . import _lib
        self.lib, self.check = _lib.load_library(), _lib.check
        self.dev, self.pieces = dev, pieces
        self.stream, self.copy_stream = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
        self.slots = [_BgzfSlot(pieces, dev) for _ in range(depth)]
        self.stream.wait_stream(torch.cuda.current_stream(dev))
        self.k = 0

    def _finish(self, slot):
        n, slot.n = slot.n, None
        slot.done.synchronize()
        lens, status = slot.host_meta[:n].numpy().view(np.uint32).copy(), slot.host_meta[self.pieces:self.pieces + n].numpy()
        bad = np.flatnonzero(status != 0)
        if len(bad):
            raise RuntimeError(f"BGZF block {int(bad[0])} of a batch: GPU deflate failed with status {int(status[bad[0]])}")
        total = int(lens.sum(dtype=np.uint64))
        with torch.cuda.device(self.dev), torch.cuda.stream(self.copy_stream):
            self.copy_stream.wait_event(slot.done)
            slot.host_out[:total].copy_(slot.packed[:total], non_blocking=True)
        self.copy_stream.synchronize()
        return slot.host_out[:total].numpy().tobytes(), lens

    def submit(self, data):
        """Queue len(data) <= pieces * 65280 bytes; -> the (blocks, lengths) of the batch this slot held before, or None."""
        slot = self.slots[self.k % len(self.slots)]
        self.k += 1
        prev = self._finish(slot) if slot.n is not None else None
        nbytes = len(data)
        n = -(-nbytes // BGZF_MAX_INPUT)
        slot.host_in[:nbytes].numpy()[:] = np.frombuffer(data, np.uint8)
        with torch.cuda.device(self.dev), torch.cuda.stream(self.stream):
            slot.dev_in[:nbytes].copy_(slot.host_in[:nbytes], non_blocking=True)
            st = self.stream.cuda_stream
            self.check(self.lib.dan_bgzf_compress_device(slot.dev_in.data_ptr(), nbytes, slot.slots.data_ptr(), slot.meta.data_ptr(),
                                                         slot.meta.data_ptr() + 4 * self.pieces, st), "dan_bgzf_compress_device")
            self.check(self.lib.dan_bgzf_compact(slot.slots.data_ptr(), slot.meta.data_ptr(), n, slot.packed.data_ptr(), slot.offsets.data_ptr(), st),
                       "dan_bgzf_compact")
            slot.host_meta.copy_(slot.meta, non_blocking=True)
            slot.done.record(self.stream)
        slot.n = n
        return prev

    def drain(self):
        """The blocks of every batch still in flight, oldest first."""
        out = []
        for j in range(len(self.slots)):
            slot = self.slots[(self.k + j) % len(self.slots)]
            if slot.n is not None:
                out.append(self._finish(slot))
        return out

    def close(self):
        self.stream.synchronize()
        self.copy_stream.synchronize()


# ---- VCF header and record checks ------------------------------------------------------------------------------------------------
def read_vcf_header(header) -> str:
    """The header text: `header` itself when it holds newlines or starts with '#', else the leading '#' lines of the VCF at that path.
    It must end with a '#CHROM' line; the result ends with one newline."""
    if isinstance(header, bytes):
        header = header.decode()
    if isinstance(header, os.PathLike) or (header and "\n" not in header and not header.startswith("#")):
        lines = []
        with open(os.fspath(header)) as f:
            for line in f:
                if not line.startswith("#"):
                    break
                lines.append(line)
        header = "".join(lines)
    lines = header.rstrip("\n").split("\n") if header.strip() else []
    if not lines or not lines[-1].startswith("#CHROM"):
        raise ValueError("a VCF header must end with its '#CHROM' line")
    bad = [l for l in lines if not l.startswith("#")]
    if bad:
        raise ValueError(f"header line {bad[0][:60]!r} does not start with '#'")
    return "\n".join(lines) + "\n"


def header_contigs(header: str) -> list:
    """The IDs of the header's ##contig=<ID=...> lines, in order."""
    return re.findall(r"^##contig=<(?:[^>]*,)?ID=([^,>]+)", header, re.M)


def record_interval(line: str):
    """(CHROM, POS, beg, end) of a VCF line: beg = POS - 1 and end = beg + len(REF), or END of the INFO column when it has that key
    (as htslib takes it), at least beg + 1. ValueError for fewer than 8 columns or a non-integer POS or END."""
    f = line.split("\t", 8)
    if len(f) < 8:
        raise ValueError(f"VCF line with {len(f)} tab-separated columns, fewer than 8: {line[:80]!r}")
    try:
        pos = int(f[1])
    except ValueError:
        raise ValueError(f"VCF line with a non-integer POS {f[1]!r}: {line[:80]!r}") from None
    beg = pos - 1
    end = beg + len(f[3])
    info = f[7]
    if "END=" in info:
        for kv in info.split(";"):
            if kv.startswith("END="):
                try:
                    end = int(kv[4:])
                except ValueError:
                    raise ValueError(f"VCF line with a non-integer END {kv[4:]!r}: {line[:80]!r}") from None
                break
    return f[0], pos, beg, max(end, beg + 1)


# ---- the .tbi index ---------------------------------------------------------------------------------------------------------------
def reg2bin(beg: int, end: int) -> int:
    """The UCSC / SAM binning scheme's smallest bin holding [beg, end): levels of 2^14, 2^17, 2^20, 2^23 and 2^26 bases."""
    end -= 1
    for shift, first in ((14, 4681), (17, 585), (20, 73), (23, 9), (26, 1)):
        if beg >> shift == end >> shift:
            return first + (beg >> shift)
    return 0


def _reg2bin_np(beg, end):
    end = end - 1
    out = np.zeros(len(beg), np.int64)
    done = np.zeros(len(beg), bool)
    for shift, first in ((14, 4681), (17, 585), (20, 73), (23, 9), (26, 1)):
        hit = ~done & ((beg >> shift) == (end >> shift))
        out[hit] = first + (beg[hit] >> shift)
        done |= hit
    return out


def build_tabix_index(names, ref_id, beg, end, vstart, vend) -> bytes:
    """The uncompressed .tbi (format 2 = VCF, col_seq 1, col_beg 2, col_end 0, meta '#', skip 0) of records in file order: record i
    lies on reference names[ref_id[i]] over [beg[i], end[i]) and occupies the virtual offsets [vstart[i], vend[i]) (block file offset
    << 16 | offset in the block). Per reference, records are contiguous and sorted by beg. Rules:
      bins     reg2bin(beg, end), ascending; consecutive records in one bin form one chunk [first vstart, last vend);
      linear   one entry per 16 kb window up to the last window a record covers: the smallest vstart of a record overlapping the
               window; an empty window takes the previous entry, windows before the first record that record's vstart;
      pseudo-bin 37450: chunk (first vstart, last vend) and chunk (record count, 0)."""
    ref_id, beg, end = (np.asarray(a, np.int64) for a in (ref_id, beg, end))
    vstart, vend = np.asarray(vstart, np.uint64), np.asarray(vend, np.uint64)
    nm = b"".join(n.encode() + b"\0" for n in names)
    out = [b"TBI\x01", struct.pack("<8i", len(names), 2, 1, 2, 0, ord("#"), 0, len(nm)), nm]
    bins_all = _reg2bin_np(beg, end)
    bounds = np.searchsorted(ref_id, np.arange(len(names) + 1))
    for r in range(len(names)):
        lo, hi = int(bounds[r]), int(bounds[r + 1])
        b, vs, ve = bins_all[lo:hi], vstart[lo:hi], vend[lo:hi]
        cut = np.flatnonzero(np.diff(b)) + 1                          # chunk starts: a record whose bin differs from its predecessor's
        first = np.concatenate(([0], cut))
        last = np.concatenate((cut, [hi - lo])) - 1
        cb, cs, ce = b[first], vs[first], ve[last]
        order = np.argsort(cb, kind="stable")                          # bins ascending, chunks of a bin in file order
        cb, cs, ce = cb[order], cs[order], ce[order]
        ubins, ustart = np.unique(cb, return_index=True)
        out.append(struct.pack("<i", len(ubins) + 1))
        for k, bn in enumerate(ubins):
            a = int(ustart[k])
            z = int(ustart[k + 1]) if k + 1 < len(ubins) else len(cb)
            out.append(struct.pack("<Ii", int(bn), z - a))
            out.append(np.stack([cs[a:z], ce[a:z]], 1).astype("<u8").tobytes())
        out.append(struct.pack("<Ii", _PSEUDO_BIN, 2) + struct.pack("<4Q", int(vs[0]), int(ve[-1]), hi - lo, 0))
        w0, w1 = beg[lo:hi] >> 14, (end[lo:hi] - 1) >> 14
        nwin = int(w1.max()) + 1
        cnt = w1 - w0 + 1
        rec = np.repeat(np.arange(hi - lo), cnt)
        win = np.repeat(w0, cnt) + (np.arange(int(cnt.sum())) - np.repeat(np.cumsum(cnt) - cnt, cnt))
        first_rec = np.full(nwin, hi - lo, np.int64)
        np.minimum.at(first_rec, win, rec)                            # vstart grows with the record index: the first record is the smallest
        filled = first_rec < hi - lo
        src = np.maximum.accumulate(np.where(filled, np.arange(nwin), -1))
        lin = np.where(src >= 0, first_rec[np.maximum(src, 0)], 0)     # empty windows: the previous entry; leading ones: record 0
        out.append(struct.pack("<i", nwin) + vs[lin].astype("<u8").tobytes())
    out.append(struct.pack("<Q", 0))
    return b"".join(out)


def parse_tabix_index(data: bytes) -> dict:
    """An uncompressed .tbi -> {"header": 7 ints, "names": [...], "refs": [{"bins": {bin: [(beg, end), ...]}, "linear": [...]}],
    "n_no_coor": int}. What concat_vcf_shards merges."""
    if data[:4] != b"TBI\x01":
        raise ValueError("not a tabix index (magic)")
    n_ref, *hdr, l_nm = struct.unpack_from("<8i", data, 4)
    p = 36
    names = data[p:p + l_nm].split(b"\0")[:-1]
    p += l_nm
    refs = []
    for _ in range(n_ref):
        (n_bin,) = struct.unpack_from("<i", data, p); p += 4
        bins = {}
        for _ in range(n_bin):
            bn, n_chunk = struct.unpack_from("<Ii", data, p); p += 8
            bins[bn] = [tuple(c) for c in np.frombuffer(data, "<u8", 2 * n_chunk, p).reshape(-1, 2).tolist()]
            p += 16 * n_chunk
        (n_intv,) = struct.unpack_from("<i", data, p); p += 4
        refs.append({"bins": bins, "linear": np.frombuffer(data, "<u8", n_intv, p).tolist()})
        p += 8 * n_intv
    n_no_coor = struct.unpack_from("<Q", data, p)[0] if p + 8 <= len(data) else 0
    return {"header": hdr, "names": [n.decode() for n in names], "refs": refs, "n_no_coor": n_no_coor}


def write_tabix_index(idx: dict) -> bytes:
    """parse_tabix_index's dict -> the uncompressed .tbi."""
    nm = b"".join(n.encode() + b"\0" for n in idx["names"])
    out = [b"TBI\x01", struct.pack("<8i", len(idx["names"]), *idx["header"], len(nm)), nm]
    for ref in idx["refs"]:
        out.append(struct.pack("<i", len(ref["bins"])))
        for bn in sorted(ref["bins"]):
            ch = ref["bins"][bn]
            out.append(struct.pack("<Ii", bn, len(ch)) + np.asarray(ch, "<u8").reshape(-1, 2).tobytes())
        out.append(struct.pack("<i", len(ref["linear"])) + np.asarray(ref["linear"], "<u8").tobytes())
    out.append(struct.pack("<Q", idx["n_no_coor"]))
    return b"".join(out)


# ---- the writer --------------------------------------------------------------------------------------------------------------------
class BgzfVcfWriter:
    """Write a VCF as BGZF (`path`, conventionally *.vcf.gz) and, with index=True, its tabix index (`path + ".tbi"`).

    header: the '##' lines and the '#CHROM' line as text, or the path of a VCF whose leading '#' lines are used (read_vcf_header);
    written into blocks of its own before the first record. write(lines) appends records (str, without or with a trailing newline);
    they must come in the order a tabix index needs: one contiguous run per CHROM, POS non-decreasing within it, and every interval
    (record_interval) below 2^29. A line that breaks this, has fewer than 8 columns or a non-integer POS raises ValueError naming it.

    The record text is cut into 65280-byte pieces whatever the line boundaries, with a carry across write() calls, so the file's
    bytes depend only on the header and the lines, not on how the lines were batched. Each piece is one BGZF block:
      device=None            host zlib raw DEFLATE at `level` (default 6) and zlib.crc32;
      device=<CUDA device>   the GPU deflate kernel (dan_bgzf_compress_device), which has one setting: `level` raises ValueError.
                             Batches of up to one piece per SM go through two rotating pinned slots, so formatting the next batch
                             on the host overlaps the GPU's work on this one.
    close() appends the 28-byte empty EOF block and builds the index on the host from the records' uncompressed offsets and the
    blocks' lengths."""

    def __init__(self, path, header, device=None, level=None, index=True, batch_pieces=None):
        self.path = os.fspath(path)
        self.header = read_vcf_header(header)
        if device is None:
            self._dev = None
            self._level = 6 if level is None else int(level)
        else:
            dev = torch.device(device)
            if dev.type != "cuda":
                raise ValueError(f"device must be a CUDA device, not {dev}")
            if level is not None:
                raise ValueError("level applies to host compression (device=None); the GPU deflate has one setting")
            if dev.index is None:
                dev = torch.device("cuda", torch.cuda.current_device())
            self._dev = dev
            pieces = batch_pieces or torch.cuda.get_device_properties(dev).multi_processor_count
            self._gpu = _DeviceBgzf(dev, pieces)
        self.index = index
        self.index_seconds = 0.0                     # host time of close()'s index build and write
        self._f = open(self.path, "wb")
        self._closed = False
        self._carry = bytearray()
        self._block_lens = array.array("q")          # data blocks, in file order
        self._names, self._name_ids = [], {}
        self._ref, self._beg, self._end, self._ustart = (array.array("q") for _ in range(4))
        self._last = None                            # (ref id, POS) of the last record
        self._ubytes = 0                             # record text bytes so far
        try:
            for blk in self._compress_now(self.header.encode()):
                self._f.write(blk)
            self.data_start = self._f.tell()
        except BaseException:
            self._abort()
            raise

    def __enter__(self):
        return self

    def __exit__(self, exc_type, exc, tb):
        if exc_type is None:
            self.close()
        else:
            self._abort()

    def _abort(self):
        if not self._closed:
            self._closed = True
            if self._dev is not None:
                self._gpu.close()
            self._f.close()

    def _compress_now(self, data):
        """data -> its blocks, synchronously (the header, and the last partial piece)."""
        if self._dev is None:
            return host_bgzf_blocks(data, self._level)
        if not data:
            return []
        blocks, offsets, lengths, _ = bgzf_compress_device(torch.from_numpy(np.frombuffer(bytes(data), np.uint8).copy()).to(self._dev))
        blob, off, ln = blocks.cpu().numpy().tobytes(), offsets.cpu().numpy(), lengths.cpu().numpy()
        return [blob[o:o + n] for o, n in zip(off, ln)]

    def _emit(self, blob, lens):
        self._f.write(blob)
        self._block_lens.extend(int(x) for x in lens)

    def write(self, lines):
        """Append VCF record lines (an iterable of str)."""
        if self._closed:
            raise ValueError("write to a closed BgzfVcfWriter")
        lines = [l[:-1] if l.endswith("\n") else l for l in lines]
        if not lines:
            return
        ids, last = self._name_ids, self._last
        for line in lines:
            chrom, pos, beg, end = record_interval(line)
            rid = ids.get(chrom)
            if rid is None:
                rid = ids[chrom] = len(self._names)
                self._names.append(chrom)
            elif last is not None and (rid != last[0] or pos < last[1]):
                what = f"contig {chrom!r} revisited" if rid != last[0] else f"POS {pos} after {last[1]}"
                raise ValueError(f"records out of order ({what}): {line[:80]!r}")
            if pos < 1 or end > TBI_MAX_POS - 1:
                raise ValueError(f"record outside the .tbi range 1 <= POS, end < 2^29 (a CSI index would be needed): {line[:80]!r}")
            last = (rid, pos)
            self._ref.append(rid); self._beg.append(beg); self._end.append(end)
        self._last = last
        text = ("\n".join(lines) + "\n").encode()
        if len(text) == sum(map(len, lines)) + len(lines):
            sizes = np.fromiter(map(len, lines), np.int64, len(lines)) + 1
        else:                                                        # non-ASCII text: byte lengths per line
            sizes = np.fromiter((len(l.encode()) + 1 for l in lines), np.int64, len(lines))
        starts = self._ubytes + np.concatenate(([0], np.cumsum(sizes)[:-1]))
        self._ustart.extend(starts.tolist())
        self._ubytes += len(text)
        self._carry += text
        self._push(final=False)

    def _push(self, final):
        """Compress the carry's whole pieces (and with `final` its partial last piece)."""
        if self._dev is None:
            n = len(self._carry) if final else len(self._carry) - len(self._carry) % BGZF_MAX_INPUT
            if n:
                blocks = host_bgzf_blocks(memoryview(self._carry)[:n], self._level)
                self._emit(b"".join(blocks), [len(b) for b in blocks])
                del self._carry[:n]
            return
        cap = self._gpu.pieces * BGZF_MAX_INPUT
        while len(self._carry) >= cap or (final and self._carry):
            n = min(cap, len(self._carry))
            done = self._gpu.submit(memoryview(self._carry)[:n])
            del self._carry[:n]
            if done is not None:
                self._emit(*done)
        if final:
            for done in self._gpu.drain():
                self._emit(*done)

    def close(self):
        """Flush the last piece, write the EOF block and, with index=True, the .tbi."""
        if self._closed:
            return
        try:
            self._push(final=True)
            self._f.write(BGZF_EOF)
        finally:
            self._abort()
        if self.index:
            t0 = time.perf_counter()
            idx = build_tabix_index(self._names, self._ref, self._beg, self._end, *self.virtual_offsets())
            with open(self.path + ".tbi", "wb") as f:
                f.write(b"".join(host_bgzf_blocks(idx, 6)) + BGZF_EOF)
            self.index_seconds = time.perf_counter() - t0

    def virtual_offsets(self):
        """(vstart, vend) of every record written, from the uncompressed offsets and the data blocks' lengths. An offset at the end of
        a block is the next block's start, as htslib reports it after reading that block's last byte."""
        lens = np.frombuffer(self._block_lens, np.int64)
        block_off = self.data_start + np.concatenate(([0], np.cumsum(lens)))
        u = np.frombuffer(self._ustart, np.int64)
        b = u // BGZF_MAX_INPUT
        v = (block_off[b].astype(np.uint64) << np.uint64(16)) | (u - b * BGZF_MAX_INPUT).astype(np.uint64)
        v = np.concatenate((v, [np.uint64(int(block_off[-1]) << 16)]))     # the end of the data: the next block's start
        return v[:-1], v[1:]


# ---- scored VCF from a record file -------------------------------------------------------------------------------------------------
def write_scored_vcf(path, model, records, header, start=0, stop=None, sort=False, device="model", index=True, **call_options) -> int:
    """call_record_file(model, records, start, stop, **call_options) into a BgzfVcfWriter(path, header, device): the scored VCF lines
    as a `.vcf.gz` with its `.tbi`. Returns the number of lines written. `failed`, `strict`, `thresholds` and the other options pass
    through unchanged. device="model" compresses on the model's GPU, None with host zlib.

    sort=False writes the lines in file order, which must already be the index's order (BgzfVcfWriter raises otherwise); sort=True
    holds the lines in memory and stably sorts them by (contig rank, POS) first, the rank following the header's ##contig lines where
    they name the contig, else first appearance. The record file guarantees no order."""
    from .feeder import call_record_file
    if isinstance(device, str) and device == "model":
        device = model._device()
    hdr = read_vcf_header(header)
    held, count = [], 0
    with BgzfVcfWriter(path, hdr, device=device, index=index) as w:
        for _names, lines, _gt, _q in call_record_file(model, records, start=start, stop=stop, **call_options):
            if sort:
                held.extend(lines)
            else:
                w.write(lines)
            count += len(lines)
        if sort:
            w.write(sort_vcf_lines(held, header_contigs(hdr)))
    return count


def sort_vcf_lines(lines, contigs=()) -> list:
    """lines stably sorted by (contig rank, POS): contigs in the order of `contigs`, then the others in order of first appearance."""
    rank = {c: k for k, c in enumerate(contigs)}
    keyed = []
    for line in lines:
        chrom, pos, _, _ = record_interval(line)
        r = rank.get(chrom)
        if r is None:
            r = rank[chrom] = len(rank)
        keyed.append((r, pos))
    order = sorted(range(len(lines)), key=keyed.__getitem__)
    return [lines[k] for k in order]


# ---- per-rank shards into one file -----------------------------------------------------------------------------------------------
def _block_spans(f):
    """[(file offset, size)] of the BGZF blocks of an open file, from their headers."""
    spans, off = [], 0
    f.seek(0, 2)
    size = f.tell()
    while off < size:
        f.seek(off)
        h = f.read(18)
        if len(h) < 18 or h[:4] != b"\x1f\x8b\x08\x04" or h[10:16] != b"\x06\0BC\x02\0":
            raise ValueError(f"{f.name}: no BGZF block at offset {off}")
        bsize = struct.unpack_from("<H", h, 16)[0] + 1
        spans.append((off, bsize))
        off += bsize
    if off != size:
        raise ValueError(f"{f.name}: the last block runs past the file's end")
    return spans


def _inflate_block(f, off, size):
    f.seek(off)
    blk = f.read(size)
    return zlib.decompressobj(-15).decompress(blk[18:-8])


class _Shard:
    """What concat_vcf_shards needs of one file: its header text, the span of its data blocks, its first and last record and its
    index."""

    def __init__(self, path):
        self.path = os.fspath(path)
        with open(self.path, "rb") as f:
            spans = _block_spans(f)
            f.seek(-len(BGZF_EOF), 2)
            if not spans or spans[-1][1] != len(BGZF_EOF) or f.read() != BGZF_EOF:
                raise ValueError(f"{self.path}: does not end with the BGZF EOF block")
            text, k = b"", 0
            while k < len(spans) - 1:                                 # the header's blocks: text up to the end of the '#CHROM' line
                text += _inflate_block(f, *spans[k])
                k += 1
                m = re.search(rb"(^|\n)#CHROM[^\n]*\n", text)
                if m:
                    break
            if not m or m.end() != len(text):
                raise ValueError(f"{self.path}: not written by BgzfVcfWriter (the data does not start on a block boundary after the header)")
            self.header = text
            self.data_start, self.data_end = spans[k][0], spans[-1][0]
            self.first = self.last = None
            if k < len(spans) - 1:
                head = _inflate_block(f, *spans[k])
                self.first = record_interval(head[:head.index(b"\n")].decode())
                tail, j = b"", len(spans) - 1
                while j > k and tail.count(b"\n") < 2:
                    j -= 1
                    tail = _inflate_block(f, *spans[j]) + tail
                self.last = record_interval(tail.rstrip(b"\n").rsplit(b"\n", 1)[-1].decode())
        with open(self.path + ".tbi", "rb") as f:
            self.index = parse_tabix_index(gzip.decompress(f.read()))


def concat_vcf_shards(path, shard_paths, index=True):
    """Join files written by BgzfVcfWriter (each rank's contiguous record range, in rank order) into one file and index without
    recompressing: the header blocks of the first shard, the data blocks of every shard as they are, one EOF block. Each shard's
    index moves by (its new data start - its old one) << 16 and merges into one per reference: bins take the chunks of every shard
    in order, the linear index takes each window from the first shard that has it. ValueError when the headers differ, a shard's
    first record sorts before the previous shard's last one (or revisits an earlier contig), or a file is not one this writer made."""
    import shutil
    shards = [_Shard(p) for p in shard_paths]
    if not shards:
        raise ValueError("no shards to concatenate")
    for s in shards[1:]:
        if s.header != shards[0].header:
            raise ValueError(f"{s.path}: its header differs from {shards[0].path}'s")
    merged = {"header": [2, 1, 2, 0, ord("#"), 0], "names": [], "refs": [], "n_no_coor": 0}
    prev = None                                                       # the last non-empty shard
    out_off = shards[0].data_start
    with open(os.fspath(path), "wb") as out:
        with open(shards[0].path, "rb") as f:
            shutil.copyfileobj(_Range(f, 0, shards[0].data_start), out)
        for s in shards:
            if s.first is not None and prev is not None:
                continues = s.first[0] == prev.last[0]
                if (continues and s.first[1] < prev.last[1]) or (not continues and s.first[0] in merged["names"]):
                    raise ValueError(f"{s.path}: its first record ({s.first[0]}:{s.first[1]}) sorts before the previous shard's last "
                                     f"({prev.last[0]}:{prev.last[1]})")
            shift = (out_off - s.data_start) << 16
            for name, ref in zip(s.index["names"], s.index["refs"]):
                bins = {bn: [(b + shift, e + shift) for b, e in ch] for bn, ch in ref["bins"].items() if bn != _PSEUDO_BIN}
                (pb, pe), (count, _) = ref["bins"][_PSEUDO_BIN]                # (first start, last end), (records, 0)
                lin = [v + shift for v in ref["linear"]]
                if name not in merged["names"]:
                    bins[_PSEUDO_BIN] = [(pb + shift, pe + shift), (count, 0)]
                    merged["names"].append(name)
                    merged["refs"].append({"bins": bins, "linear": lin})
                    continue
                if name != merged["names"][-1]:
                    raise ValueError(f"{s.path}: contig {name!r} revisited")
                tgt = merged["refs"][-1]
                (b0, _), (n0, _) = tgt["bins"][_PSEUDO_BIN]
                tgt["bins"][_PSEUDO_BIN] = [(b0, pe + shift), (n0 + count, 0)]
                for bn, ch in bins.items():
                    tgt["bins"].setdefault(bn, []).extend(ch)
                tgt["linear"].extend(lin[len(tgt["linear"]):])
            with open(s.path, "rb") as f:
                shutil.copyfileobj(_Range(f, s.data_start, s.data_end), out)
            out_off += s.data_end - s.data_start
            if s.first is not None:
                prev = s
        out.write(BGZF_EOF)
    if index:
        with open(os.fspath(path) + ".tbi", "wb") as f:
            f.write(b"".join(host_bgzf_blocks(write_tabix_index(merged), 6)) + BGZF_EOF)


class _Range:
    """A file's bytes [lo, hi) as a readable object for shutil.copyfileobj."""

    def __init__(self, f, lo, hi):
        self.f, self.left = f, hi - lo
        f.seek(lo)

    def read(self, n=-1):
        n = self.left if n < 0 else min(n, self.left)
        self.left -= n
        return self.f.read(n)
