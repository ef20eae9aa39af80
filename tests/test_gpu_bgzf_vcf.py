"""BGZF VCF output: BGZF blocks field by field (host writer on the CPU, `dan_bgzf_compress_device` on the GPU), the cut into 65280-byte
pieces whatever the batching, the .tbi checked through this file's own parser and region query against a linear scan, the order
checks, sorting, shard concatenation, the C argument checks, the pinned bytes of `dan_deflate_device`, and write_scored_vcf end to end.

The index reader here restates the SAM/tabix specification (reg2bins, the linear-index lower bound, a seek by virtual offset) and
shares no code with dl4vc_b200.vcf. Neither htslib nor tabix is available to the suite, so conformance with them rests on the
specification and on this reader."""
import ctypes as C
import gzip
import hashlib
import os
import random
import struct
import sys
import zlib

import numpy as np
import pytest
import torch

from test_gpu_record_calls import DEPTHS, make_records
from dl4vc_b200.vcf import (BGZF_EOF, BgzfVcfWriter, build_tabix_index, concat_vcf_shards, read_vcf_header, sort_vcf_lines,
                            write_scored_vcf)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PIECE = 65280
HEADER = ("##fileformat=VCFv4.2\n##contig=<ID=chrB>\n##contig=<ID=chrA>\n##contig=<ID=chrS>\n"
          "#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\tS\n")


# ---- an independent BGZF / .tbi reader ----------------------------------------------------------------------------------------------
def blocks(data):
    """[(offset, size, raw deflate, crc, isize)] of a BGZF file, every header field checked."""
    out, p = [], 0
    while p < len(data):
        id1, id2, cm, flg, mtime, xfl, os_, xlen, si1, si2, slen, bsize = struct.unpack_from("<BBBBIBBHBBHH", data, p)
        assert (id1, id2, cm, flg, mtime, xfl, os_, xlen, si1, si2, slen) == (31, 139, 8, 4, 0, 0, 255, 6, 66, 67, 2), p
        size = bsize + 1
        crc, isize = struct.unpack_from("<II", data, p + size - 8)
        out.append((p, size, data[p + 18:p + size - 8], crc, isize))
        p += size
    assert p == len(data)
    return out


def inflate(raw):
    d = zlib.decompressobj(-15)
    out = d.decompress(raw) + d.flush()
    assert d.eof and not d.unused_data
    return out


def check_blocks(data):
    """Every block valid; -> (the inflated pieces, block sizes). The file ends with the EOF block."""
    assert data.endswith(BGZF_EOF)
    pieces, sizes = [], []
    for off, size, raw, crc, isize in blocks(data):
        text = inflate(raw)
        assert crc == zlib.crc32(text) and isize == len(text), off
        pieces.append(text)
        sizes.append(size)
    return pieces, sizes


def parse_tbi(path):
    d = gzip.decompress(open(path, "rb").read())
    assert d[:4] == b"TBI\x01"
    n_ref, fmt, col_seq, col_beg, col_end, meta, skip, l_nm = struct.unpack_from("<8i", d, 4)
    p = 36
    names = [n.decode() for n in d[p:p + l_nm].split(b"\0")[:-1]]
    p += l_nm
    refs = []
    for _ in range(n_ref):
        (n_bin,) = struct.unpack_from("<i", d, p); p += 4
        bins = {}
        for _ in range(n_bin):
            b, nc = struct.unpack_from("<Ii", d, p); p += 8
            bins[b] = [struct.unpack_from("<QQ", d, p + 16 * k) for k in range(nc)]
            p += 16 * nc
        (n_intv,) = struct.unpack_from("<i", d, p); p += 4
        refs.append((bins, list(struct.unpack_from(f"<{n_intv}Q", d, p))))
        p += 8 * n_intv
    (n_no_coor,) = struct.unpack_from("<Q", d, p)
    assert p + 8 == len(d)
    return dict(n_ref=n_ref, fields=(fmt, col_seq, col_beg, col_end, meta, skip), names=names, refs=refs, n_no_coor=n_no_coor)


def reg2bins(beg, end):
    end -= 1
    out = [0]
    for shift, first in ((26, 1), (23, 9), (20, 73), (17, 585), (14, 4681)):
        out += range(first + (beg >> shift), first + (end >> shift) + 1)
    return out


def interval(line):
    f = line.split("\t")
    beg = int(f[1]) - 1
    end = beg + len(f[3])
    for kv in f[7].split(";"):
        if kv.startswith("END="):
            end = int(kv[4:])
    return f[0], beg, max(end, beg + 1)


class Reader:
    """Region queries through the index: the bins of the region, chunks cut by the linear index, a seek by virtual offset."""

    def __init__(self, path):
        self.data = open(path, "rb").read()
        self.idx = parse_tbi(path + ".tbi")
        self.cache = {}

    def block(self, off):
        if off not in self.cache:
            (bsize,) = struct.unpack_from("<H", self.data, off + 16)
            self.cache[off] = (inflate(self.data[off + 18:off + bsize + 1 - 8]), off + bsize + 1)
        return self.cache[off]

    def lines_from(self, v, stop):
        """(line, start voffset) from v until the voffset reaches stop."""
        off, within = v >> 16, v & 0xffff
        while (off << 16 | within) < stop:
            text, nxt = self.block(off)
            if within >= len(text):
                off, within = nxt, 0
                continue
            start, buf = off << 16 | within, b""
            while True:
                text, nxt = self.block(off)
                j = text.find(b"\n", within)
                if j >= 0:
                    buf += text[within:j]
                    within = j + 1
                    break
                buf += text[within:]
                off, within = nxt, 0
            yield buf.decode(), start

    def query(self, chrom, beg, end):
        if chrom not in self.idx["names"]:
            return []
        bins, lin = self.idx["refs"][self.idx["names"].index(chrom)]
        w = beg >> 14
        min_off = lin[w] if w < len(lin) else (lin[-1] if lin else 0)
        chunks = sorted(c for b in reg2bins(beg, end) for c in bins.get(b, ()) if c[1] > min_off)
        seen, out = set(), []
        for cb, ce in chunks:
            for line, v in self.lines_from(cb, ce):
                c, b, e = interval(line)
                if c == chrom and b < end and e > beg and v not in seen:
                    seen.add(v)
                    out.append((v, line))
        return [l for _, l in sorted(out)]


def scan(text, chrom, beg, end):
    out = []
    for line in text.split("\n"):
        if line and not line.startswith("#"):
            c, b, e = interval(line)
            if c == chrom and b < end and e > beg:
                out.append(line)
    return out


# ---- synthetic VCFs ----------------------------------------------------------------------------------------------------------------
def _line(chrom, pos, ref_len, rng, info="DP=7"):
    return f"{chrom}\t{pos}\tBP=0.{rng.randrange(10**8):08d}\t{'ACGT'[pos % 4] * ref_len}\tG\t50\t.\t{info}\tGT\t0/1"


def index_vcf(seed=1):
    """Three contigs, one with a single record; positions at and around multiples of 2^14 .. 2^26 and up to 2^29 - 1; REF of 1-300;
    400 records in one 16 kb window; one record with END=."""
    rng = random.Random(seed)
    pos = set()
    for s in (14, 17, 20, 23, 26):
        for k in range(1, 5):
            for d in (-301, -2, -1, 0, 1, 2, 150):
                p = k * (1 << s) + d
                if 1 <= p < (1 << 29) - 300:
                    pos.add(p)
    pos |= {rng.randrange(1, (1 << 29) - 300) for _ in range(1500)}
    pos |= {5 * (1 << 14) + rng.randrange(16000) for _ in range(400)}
    lines = []
    for p in sorted(pos):
        lines.append(_line("chrB", p, rng.randint(1, 300) if rng.random() < 0.3 else 1, rng))
        if rng.random() < 0.1:
            lines.append(_line("chrB", p, rng.randint(1, 300), rng))                       # a tie at the same POS
    lines.append(_line("chrB", (1 << 29) - 1, 1, rng))
    k = len(lines) // 2
    lines.insert(k, _line("chrB", int(lines[k].split("\t")[1]), 1, rng, info=f"END={int(lines[k].split(chr(9))[1]) + 150000};DP=3"))
    lines.append(_line("chrS", 777, 5, rng))
    for p in sorted(rng.randrange(1, 3 << 20) for _ in range(600)):
        lines.append(_line("chrA", p, rng.randint(1, 40), rng))
    return lines


def write_host(path, lines, batches=None, **kw):
    with BgzfVcfWriter(path, HEADER, **kw) as w:
        if batches is None:
            w.write(lines)
        else:
            lo = 0
            for n in batches:
                w.write(lines[lo:lo + n])
                lo += n
            w.write(lines[lo:])
    return open(path, "rb").read()


# ---- CPU: the host writer ------------------------------------------------------------------------------------------------------
def test_host_writer_whole_file_and_blocks(tmp_path):
    lines = index_vcf()
    data = write_host(str(tmp_path / "a.vcf.gz"), lines)
    body = "\n".join(lines) + "\n"
    assert gzip.decompress(data).decode() == HEADER + body
    pieces, sizes = check_blocks(data)
    k, acc = 0, b""
    while acc != HEADER.encode():                                   # the header sits in blocks of its own
        acc += pieces[k]
        k += 1
        assert len(acc) <= len(HEADER)
    data_pieces = pieces[k:-1]
    assert len(data_pieces) > 3 and all(len(p) == PIECE for p in data_pieces[:-1]) and 0 < len(data_pieces[-1]) <= PIECE
    assert b"".join(data_pieces).decode() == body
    assert pieces[-1] == b"" and data[-28:] == BGZF_EOF


def test_feeding_does_not_change_the_bytes(tmp_path):
    lines = index_vcf(seed=2)
    whole = write_host(str(tmp_path / "a.vcf.gz"), lines)
    one = write_host(str(tmp_path / "b.vcf.gz"), lines, batches=[1] * len(lines))
    rng = random.Random(3)
    rand = write_host(str(tmp_path / "c.vcf.gz"), lines, batches=[rng.randint(0, 700) for _ in range(20)])
    assert whole == one == rand
    assert open(tmp_path / "a.vcf.gz.tbi", "rb").read() == open(tmp_path / "c.vcf.gz.tbi", "rb").read()


def _regions(rng, lines, n):
    chroms = ["chrB", "chrA", "chrS", "chrZ"]
    out = []
    for _ in range(n):
        c = rng.choice(chroms)
        if rng.random() < 0.5:                                      # near a record
            f = rng.choice(lines).split("\t")
            c, b = f[0], max(0, int(f[1]) - 1 - rng.randint(0, 20000))
        else:
            b = rng.randrange(0, 1 << 29)
        e = min(1 << 29, b + 1 + int(2 ** rng.uniform(0, 24)))
        out.append((c, b, e))
    return out


def test_index_queries_match_a_linear_scan(tmp_path):
    lines = index_vcf()
    path = str(tmp_path / "a.vcf.gz")
    data = write_host(path, lines)
    text = gzip.decompress(data).decode()
    r = Reader(path)
    rng = random.Random(9)
    hits = 0
    for c, b, e in _regions(rng, lines, 3000) + [("chrB", 0, 1 << 29), ("chrS", 0, 1 << 29), ("chrB", (1 << 29) - 2, 1 << 29)]:
        want = scan(text, c, b, e)
        assert r.query(c, b, e) == want, (c, b, e)
        hits += len(want) > 0
    assert hits > 600


def test_index_fixed_fields(tmp_path):
    lines = index_vcf()
    path = str(tmp_path / "a.vcf.gz")
    write_host(path, lines)
    idx = parse_tbi(path + ".tbi")
    assert idx["fields"] == (2, 1, 2, 0, ord("#"), 0) and idx["n_no_coor"] == 0
    assert idx["names"] == ["chrB", "chrS", "chrA"] and idx["n_ref"] == 3
    r = Reader(path)
    starts = {}
    for line, v in r.lines_from(r.idx["refs"][0][0][37450][0][0], (len(r.data) - 28) << 16):
        if line:
            starts.setdefault(line.split("\t")[0], []).append((v, interval(line)))
    for name, (bins, lin) in zip(idx["names"], idx["refs"]):
        recs = starts[name]
        pb = bins[37450]
        assert len(pb) == 2 and pb[0][0] == recs[0][0] and pb[1] == (len(recs), 0)
        assert max(b for b in bins) == 37450
        for v, (_, b, e) in recs:                                   # every linear entry bounds the records of its window from below
            for w in range(b >> 14, ((e - 1) >> 14) + 1):
                assert lin[w] <= v
        assert len(lin) == max(((e - 1) >> 14) + 1 for _, (_, b, e) in recs)
    # the pseudo-bin's end is the last record's end: the next record's start, or the EOF block for the last reference
    assert idx["refs"][-1][0][37450][0][1] >> 16 == len(open(path, "rb").read()) - 28


@pytest.mark.parametrize("bad,match", [
    (["chrA\t5\t.\tA\tG\t50\t.\t.", "chrB\t1\t.\tA\tG\t50\t.\t.", "chrA\t9\t.\tA\tG\t50\t.\t."], "revisited"),
    (["chrA\t5\t.\tA\tG\t50\t.\t.", "chrA\t4\t.\tA\tG\t50\t.\t."], "POS 4 after 5"),
    (["chrA\t5\t.\tA\tG\t50\t."], "fewer than 8"),
    (["chrA\tfive\t.\tA\tG\t50\t.\t."], "non-integer POS"),
    ([f"chrA\t{1 << 29}\t.\tA\tG\t50\t.\t."], "2\\^29"),
    (["chrA\t5\t.\tA\tG\t50\t.\tEND=536870913"], "2\\^29"),
])
def test_order_and_format_errors(tmp_path, bad, match):
    with pytest.raises(ValueError, match=match):
        with BgzfVcfWriter(str(tmp_path / "x.vcf.gz"), HEADER) as w:
            w.write(bad)


def test_header_errors_and_header_from_a_file(tmp_path):
    for bad in ("##fileformat=VCFv4.2\n", "", "##x\n#CHROM\tPOS\n##late\n"):
        with pytest.raises(ValueError, match="#CHROM"):
            BgzfVcfWriter(str(tmp_path / "x.vcf.gz"), bad)
    src = tmp_path / "in.vcf"
    src.write_text(HEADER + "chrA\t5\t.\tA\tG\t50\t.\t.\n")
    assert read_vcf_header(str(src)) == HEADER
    with pytest.raises(ValueError, match="level"):
        BgzfVcfWriter(str(tmp_path / "x.vcf.gz"), HEADER, device="cuda:0", level=6)
    with pytest.raises(ValueError, match="CUDA device"):
        BgzfVcfWriter(str(tmp_path / "x.vcf.gz"), HEADER, device="cpu")


def test_sort_follows_contig_lines_then_first_appearance_and_is_stable():
    rng = random.Random(4)
    lines = [f"{c}\t{p}\t.\tA\tG\t50\t.\tK={k}" for k, (c, p) in
             enumerate((rng.choice(["chrA", "chrB", "chrQ", "chrS", "chrP"]), rng.randint(1, 30)) for _ in range(400))]
    ordered = sort_vcf_lines(lines, ["chrB", "chrA", "chrS"])
    rank = {"chrB": 0, "chrA": 1, "chrS": 2}
    for c in (l.split("\t")[0] for l in lines):
        rank.setdefault(c, len(rank))
    key = lambda l: (rank[l.split("\t")[0]], int(l.split("\t")[1]), int(l.split("K=")[1]))
    assert ordered == sorted(lines, key=key)                        # ties keep their input order (K grows with it)
    first = []
    for l in lines:
        if l.split("\t")[0] not in first:
            first.append(l.split("\t")[0])
    assert [l.split("\t")[0] for l in sort_vcf_lines(lines)][::1] == sorted([l.split("\t")[0] for l in lines], key=first.index)


def test_concatenated_shards_equal_one_file(tmp_path):
    lines = index_vcf(seed=5)
    one = str(tmp_path / "one.vcf.gz")
    write_host(one, lines)
    cuts = [0, 700, 700, 1300, 1950, len(lines)]                     # an empty shard, and shards that split contigs
    shards = []
    for k in range(len(cuts) - 1):
        p = str(tmp_path / f"s{k}.vcf.gz")
        write_host(p, lines[cuts[k]:cuts[k + 1]])
        shards.append(p)
    cat = str(tmp_path / "cat.vcf.gz")
    concat_vcf_shards(cat, shards)
    a, b = open(one, "rb").read(), open(cat, "rb").read()
    assert gzip.decompress(a) == gzip.decompress(b)
    check_blocks(b)
    text = gzip.decompress(b).decode()
    r1, r2 = Reader(one), Reader(cat)
    assert parse_tbi(cat + ".tbi")["names"] == parse_tbi(one + ".tbi")["names"]
    for c, lo, hi in _regions(random.Random(6), lines, 1500):
        want = scan(text, c, lo, hi)
        assert r2.query(c, lo, hi) == want == r1.query(c, lo, hi), (c, lo, hi)


def test_concatenation_rejects_overlap_other_headers_and_foreign_files(tmp_path):
    lines = index_vcf(seed=7)
    a, b = str(tmp_path / "a.vcf.gz"), str(tmp_path / "b.vcf.gz")
    write_host(a, lines[:800])
    write_host(b, lines[700:])
    with pytest.raises(ValueError, match="sorts before"):
        concat_vcf_shards(str(tmp_path / "x.vcf.gz"), [a, b])
    with pytest.raises(ValueError, match="sorts before|revisited"):
        concat_vcf_shards(str(tmp_path / "x.vcf.gz"), [b, a])
    c = str(tmp_path / "c.vcf.gz")
    with BgzfVcfWriter(c, HEADER.replace("S\n", "T\n")) as w:
        w.write(lines[800:])
    with pytest.raises(ValueError, match="header differs"):
        concat_vcf_shards(str(tmp_path / "x.vcf.gz"), [a, c])
    d = str(tmp_path / "d.vcf.gz")                                   # one gzip member for header and data: not this writer's
    text = (HEADER + "\n".join(lines[800:]) + "\n").encode()
    c0 = zlib.compressobj(6, zlib.DEFLATED, -15)
    raw = c0.compress(text[:PIECE]) + c0.flush()
    with open(d, "wb") as f:
        f.write(b"\x1f\x8b\x08\x04\0\0\0\0\0\xff\x06\0BC\x02\0" + struct.pack("<H", 26 + len(raw) - 1) + raw
                + struct.pack("<II", zlib.crc32(text[:PIECE]), PIECE) + BGZF_EOF)
    open(d + ".tbi", "wb").write(open(a + ".tbi", "rb").read())
    with pytest.raises(ValueError, match="block boundary"):
        concat_vcf_shards(str(tmp_path / "x.vcf.gz"), [a, d])


# ---- CPU: C argument checks -----------------------------------------------------------------------------------------------------
def test_bgzf_entry_points_check_arguments_before_any_launch():
    """Null pointers fail and bytes = 0 succeeds without a launch, so these run without a GPU."""
    from dl4vc_b200 import _lib
    lib = _lib.load_library()
    p = C.c_void_p(16)
    f = lib.dan_bgzf_compress_device
    for args in ((None, 100, p, p, p), (p, 100, None, p, p), (p, 100, p, None, p), (p, 100, p, p, None)):
        assert f(*args, None) == -1 and b"null" in lib.dan_last_error(), args
    assert f(None, 0, None, None, None, None) == 0
    assert lib.dan_bgzf_compact(p, p, -1, p, p, None) == -1 and b"negative" in lib.dan_last_error()
    assert lib.dan_bgzf_compact(p, p, 2, p, None, None) == -1 and b"null" in lib.dan_last_error()
    assert lib.dan_bgzf_compact(None, p, 2, p, p, None) == -1 and b"null" in lib.dan_last_error()


def test_bgzf_compress_device_argument_checks():
    from dl4vc_b200.vcf import bgzf_compress_device
    for bad in (torch.zeros(8, dtype=torch.uint8), torch.zeros((2, 8), dtype=torch.uint8), np.zeros(8, np.uint8)):
        with pytest.raises(ValueError, match="CUDA uint8"):
            bgzf_compress_device(bad)


# ---- GPU: blocks of every size and kind --------------------------------------------------------------------------------------------
def _gpu_blocks(data: bytes):
    from dl4vc_b200.vcf import bgzf_compress_device
    src = torch.from_numpy(np.frombuffer(data, np.uint8).copy()).cuda()
    packed, offsets, lengths, status = bgzf_compress_device(src)
    torch.cuda.synchronize()
    st, off, ln = status.cpu().numpy(), offsets.cpu().numpy(), lengths.cpu().numpy()
    assert not st.any() and len(ln) == -(-len(data) // PIECE)
    assert np.array_equal(off, np.cumsum(ln, dtype=np.int64) - ln) and packed.numel() == ln.sum()
    blob = packed.cpu().numpy().tobytes()
    return [blob[o:o + n] for o, n in zip(off, ln)]


def _kinds(size, seed):
    rng = np.random.default_rng(seed)
    sys.path.insert(0, os.path.join(ROOT, "scripts"))
    try:
        from bench_bgzf_vcf import synthetic_scored_lines
    finally:
        sys.path.pop(0)
    text = ("\n".join(synthetic_scored_lines(max(8, size // 60), seed)) + "\n").encode()
    runs = b"".join(bytes([65 + k % 3]) * (259 + 37 * k) for k in range(size // 259 + 2))
    return {"vcf": (text * (size // max(len(text), 1) + 1))[:size], "random": rng.integers(0, 256, size, dtype=np.uint8).tobytes(),
            "zeros": bytes(size), "runs": runs[:size]}


SIZES = [0, 1, 31, 32, 33, 1023, 1024, 1025, 16383, 16384, 16385, 65279, 65280, 65281, 3 * PIECE + 17]


@pytest.mark.gpu
@pytest.mark.parametrize("size", SIZES)
def test_blocks_of_every_size_and_kind(size):
    for kind, data in _kinds(size, size).items():
        out = _gpu_blocks(data)
        for k, blk in enumerate(out):
            piece = data[k * PIECE:(k + 1) * PIECE]
            ((off, bsize, raw, crc, isize),) = blocks(blk)
            assert bsize == len(blk) <= 65536, (kind, k)
            assert inflate(raw) == piece, (kind, k)
            assert crc == zlib.crc32(piece) and isize == len(piece), (kind, k)
            if kind == "random":                                    # the stored fallback, at exactly its size
                assert len(blk) == 18 + 5 + len(piece) + 8 and raw[0] & 6 == 0, k
            elif kind != "vcf" and len(piece) >= 1024:               # zeros and long runs
                assert len(blk) < len(piece) // 8, (kind, k, len(blk))
        assert gzip.decompress(b"".join(out) + BGZF_EOF) == data, kind


@pytest.mark.gpu
def test_block_bytes_depend_only_on_their_piece(tmp_path):
    data = _kinds(5 * PIECE + 999, 3)["vcf"]
    alone = [_gpu_blocks(data[k * PIECE:(k + 1) * PIECE])[0] for k in range(6)]
    assert _gpu_blocks(data) == alone
    assert _gpu_blocks(data) == alone                                # a repeat call
    assert _gpu_blocks(data[PIECE:2 * PIECE] * 7) == [alone[1]] * 7  # the same piece at every position of a launch
    lines = index_vcf(seed=8)
    files = []
    for k, batches in enumerate((None, [1] * 500, [random.Random(2).randint(0, 900) for _ in range(15)])):
        files.append(write_host(str(tmp_path / f"g{k}.vcf.gz"), lines, batches, device="cuda:0", batch_pieces=2 + k))
    assert files[0] == files[1] == files[2]


# ---- GPU: the zlib streams of dan_deflate_device are unchanged -----------------------------------------------------------------------
# SHA-256 of (u32 stream lengths, then the packed streams) of dan_deflate_device on the inputs below, taken from the kernel before the
# BGZF container was added to it (one B200).
PINNED = {
    "records": ("bdece35aae18ad3772e5edc9acf6399bfe5032c13e8bfd4b2b994ddfc30e1e3a", 1902348),
    "text4096": ("0c75440376644eb285fa49ac615535d08b9d9a96b71611951a99a842c903b345", 27238),
    "text65537": ("a8296c4e587bcb1ee64f5252a47ec18a870d724b5cab57480702cfe01afed296", 14499),
}


def _pinned_inputs():
    recs = make_records(48, seed=2026, depths=DEPTHS, broken=(5, 30))
    rng = np.random.default_rng(2026)
    text = b"".join(b"chr%d\t%d\t.\tA\tG\t50\t.\tDP=%d\n" % (1 + k % 3, 1000 + 7 * k, rng.integers(5, 90)) for k in range(3000))
    return {"records": [r.tobytes() for r in recs.view(np.uint8).reshape(len(recs), -1)],
            "text4096": [text[k * 4096:(k + 1) * 4096] for k in range(20)], "text65537": [text[:65537]]}


@pytest.mark.gpu
def test_deflate_device_streams_are_unchanged():
    from dl4vc_b200.feeder import deflate_device
    for name, rows in _pinned_inputs().items():
        src = torch.from_numpy(np.frombuffer(b"".join(rows), np.uint8).copy().reshape(len(rows), -1)).cuda()
        streams, offsets, lengths, status = deflate_device(src)
        assert not status.cpu().numpy().any()
        h = hashlib.sha256(lengths.cpu().numpy().astype("<u4").tobytes())
        h.update(streams.cpu().numpy().tobytes())
        assert (h.hexdigest(), int(streams.numel())) == PINNED[name], name


# ---- GPU: the GPU writer against the host writer -------------------------------------------------------------------------------------
def _voffsets(data, data_start, lines):
    """(vstart, vend) of each record from the file's own block sizes."""
    sizes = [s for _, s, *_ in blocks(data)]
    starts = np.cumsum([0] + sizes)
    k = list(starts).index(data_start)
    block_off = [int(x) for x in starts[k:]]
    u = np.concatenate(([0], np.cumsum([len(l) + 1 for l in lines])))
    v = [(block_off[x // PIECE] << 16) | (x % PIECE) if x < u[-1] else block_off[-2] << 16 for x in u]
    return v[:-1], v[1:]


@pytest.mark.gpu
@pytest.mark.parametrize("seed", [1, 5])
def test_gpu_writer_against_host_writer(tmp_path, seed):
    lines = index_vcf(seed)
    g, h = str(tmp_path / "g.vcf.gz"), str(tmp_path / "h.vcf.gz")
    gd, hd = write_host(g, lines, device="cuda:0"), write_host(h, lines)
    assert gzip.decompress(gd) == gzip.decompress(hd)
    gp, gs = check_blocks(gd)
    hp, _ = check_blocks(hd)
    assert [len(p) for p in gp] == [len(p) for p in hp]
    n_header = next(k for k in range(len(gp)) if b"".join(gp[:k + 1]) == HEADER.encode()) + 1
    names, ref, beg, end = [], [], [], []
    for l in lines:
        c, b, e = interval(l)
        if c not in names:
            names.append(c)
        ref.append(names.index(c)); beg.append(b); end.append(e)
    vs, ve = _voffsets(gd, sum(gs[:n_header]), lines)
    want = build_tabix_index(names, ref, beg, end, vs, ve)
    assert gzip.decompress(open(g + ".tbi", "rb").read()) == want
    r, text = Reader(g), gzip.decompress(gd).decode()
    for c, lo, hi in _regions(random.Random(seed), lines, 300):
        assert r.query(c, lo, hi) == scan(text, c, lo, hi)


SIZE_BAR = 1.5                                                      # GPU file bytes over the host level-1 file's


@pytest.mark.gpu
def test_size_against_host_level_1(tmp_path):
    sys.path.insert(0, os.path.join(ROOT, "scripts"))
    try:
        from bench_bgzf_vcf import synthetic_scored_lines
    finally:
        sys.path.pop(0)
    lines = synthetic_scored_lines(60000, 11)
    g = len(write_host(str(tmp_path / "g.vcf.gz"), lines, device="cuda:0"))
    h = len(write_host(str(tmp_path / "h.vcf.gz"), lines, level=1))
    print(f"GPU {g / len(lines):.2f} B/line, host zlib level 1 {h / len(lines):.2f} B/line, ratio {g / h:.3f}")
    assert g <= SIZE_BAR * h, g / h


# ---- GPU: record file -> scored .vcf.gz ----------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["raw", "zlib"])
def test_write_scored_vcf_end_to_end(tmp_path, fmt):
    from dl4vc_b200.config import small_config
    from dl4vc_b200.factory import build_model
    from dl4vc_b200.feeder import call_record_file, write_compressed_records
    from dl4vc_b200.weights import synth_state_dict
    cfg = small_config()
    model = build_model(cfg, synth_state_dict(cfg, seed=3), device="cuda:0").eval()
    recs = make_records(700, seed=41, broken=(3, 300, 301))
    path = str(tmp_path / "r.bin")
    recs.tofile(path)
    if fmt == "zlib":
        cz = str(tmp_path / "r.dz")
        write_compressed_records(cz, recs, device="cuda:0")
        path = cz
    header = "##fileformat=VCFv4.2\n" + "".join(f"##contig=<ID=chr{c}>\n" for c in (3, 1, 2)) + "#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\tS\n"
    kw = dict(thresholds=dict(snp=0.4), batch_size=128, start=5, stop=690)
    fw, fc = [], []
    out = str(tmp_path / "s.vcf.gz")
    n = write_scored_vcf(out, model, path, header, sort=True, strict=False, failed=fw, **kw)
    want = [l for _, ls, _, _ in call_record_file(model, path, strict=False, failed=fc, **kw) for l in ls]
    assert fw == fc == [(300, 3), (301, 3)] and n == len(want)            # record 3 lies before `start`
    body = gzip.decompress(open(out, "rb").read()).decode()
    assert body == header + "".join(l + "\n" for l in sort_vcf_lines(want, ["chr3", "chr1", "chr2"]))
    check_blocks(open(out, "rb").read())
    r = Reader(out)
    for c, lo, hi in _regions(random.Random(2), want, 400):
        assert r.query(c, lo, hi) == scan(body, c, lo, hi)
    with pytest.raises(ValueError, match="out of order"):            # the record file is not in index order
        write_scored_vcf(str(tmp_path / "u.vcf.gz"), model, path, header, strict=False, **kw)
