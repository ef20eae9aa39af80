"""Compressed record files: the container (write / open / unpack, header pass over sidecars), the device inflate kernel
(`dan_inflate_device`) against the standard-library zlib, the compressed device decode against the host decode of the raw records,
and `call_record_file` on a compressed file against the same call on the raw file."""
import contextlib
import ctypes as C
import itertools
import os
import zlib

import numpy as np
import pytest
import torch

from test_gpu_record_calls import DEPTHS, SCALAR_KEYS, _CASES, _collect, feeder_golden, make_records
from dl4vc_b200.feeder import (RECORD_BYTES, RECORD_DTYPE, CompressedRecordFile, HostBatch, RecordFile, decode_record_headers,
                               decode_records, open_record_file, write_compressed_records)


def _raw_bytes(recs):
    return np.ascontiguousarray(recs).view(np.uint8).tobytes()


@pytest.fixture(scope="module")
def synth_pair(tmp_path_factory):
    """45 records (depths 0-200, two the loader raises on) written raw and compressed."""
    d = tmp_path_factory.mktemp("records")
    recs = make_records(45, seed=21, depths=DEPTHS, broken=(7, 30))
    raw, cz = str(d / "records.bin"), str(d / "records.dz")
    recs.tofile(raw)
    write_compressed_records(cz, recs, level=1)
    return RecordFile(raw), CompressedRecordFile(cz)


# ---- CPU: the container -----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("which", ["golden", "noise", "clean", "broken", "slices"])
def test_write_then_unpack_gives_back_the_raw_bytes(which, tmp_path):
    if which == "golden":
        recs = feeder_golden()["records"].view(RECORD_DTYPE).reshape(-1)
    else:
        recs = make_records(29, seed=4, noise_rows=which != "clean", broken=(3, 11) if which == "broken" else ())
    src = (recs[lo:lo + 6] for lo in range(0, len(recs), 6)) if which == "slices" else RecordFile(recs) if which == "clean" else recs
    path = str(tmp_path / "r.dz")
    assert write_compressed_records(path, src, level=6, threads=3) == len(recs)
    cf = open_record_file(path)
    assert isinstance(cf, CompressedRecordFile) and len(cf) == len(recs)
    cf.unpack(str(tmp_path / "r.bin"))
    with open(tmp_path / "r.bin", "rb") as f:
        assert f.read() == _raw_bytes(recs)
    sub = cf.records([len(recs) - 1, 0, 2, 0])
    assert _raw_bytes(sub) == _raw_bytes(recs[[len(recs) - 1, 0, 2, 0]])
    for name in ("name", "num_reads", "label", "vcfrec", "ref_bases", "q-scores"):
        assert np.array_equal(cf.field(2, name), recs[2][name]), name
    assert isinstance(open_record_file(str(tmp_path / "r.bin")), RecordFile)


def test_empty_source_writes_an_empty_file(tmp_path):
    path = str(tmp_path / "e.dz")
    assert write_compressed_records(path, make_records(1, seed=1)[:0]) == 0
    cf = CompressedRecordFile(path)
    assert len(cf) == 0 and cf.max_stream_bytes == 0


@pytest.mark.parametrize("max_reads,store,seed", list(itertools.product((1, 20, 100, 200), (50, 100, 200), (5, 6))))
def test_sidecar_header_pass_equals_raw_header_pass(max_reads, store, seed, tmp_path):
    recs = np.concatenate([feeder_golden()["records"].view(RECORD_DTYPE).reshape(-1), make_records(24, seed=11, depths=DEPTHS, broken=(4,))])
    path = str(tmp_path / "r.dz")
    write_compressed_records(path, recs, level=1)
    cf, rf = CompressedRecordFile(path), RecordFile(recs)
    idx = np.random.default_rng(seed).choice(len(recs), 40, replace=True)
    kw = dict(seed=seed, max_reads=max_reads, store_max_reads=store)
    got, want = decode_record_headers(cf, idx, **kw), decode_record_headers(rf, idx, **kw)
    assert np.array_equal(got[0], want[0])
    for k in SCALAR_KEYS:
        assert np.array_equal(got[1][k], want[1][k]), k
    assert np.array_equal(got[2], want[2]) and np.array_equal(got[3], want[3])
    assert (want[1]["status"] != 0).any()


def test_malformed_files_raise_on_open(tmp_path):
    recs = make_records(5, seed=2, noise_rows=False)
    path = str(tmp_path / "r.dz")
    write_compressed_records(path, recs)
    blob = open(path, "rb").read()
    h = np.frombuffer(blob[:64], np.dtype([("magic", "S8"), ("version", "<u4"), ("record_bytes", "<u4"), ("count", "<u8"), ("index_off", "<u8"),
                                           ("sidecar_off", "<u8"), ("data_off", "<u8"), ("data_bytes", "<u8"), ("sc", "<u4"), ("r", "<u4")]))[0]

    def opened(data):
        p = str(tmp_path / "bad.dz")
        with open(p, "wb") as f:
            f.write(data)
        return CompressedRecordFile(p)

    for cut in (0, 10, 63, 64, int(h["data_off"]) + 100, int(h["sidecar_off"]) + 10, len(blob) - 1):
        with pytest.raises(ValueError):
            opened(blob[:cut])
    with pytest.raises(ValueError, match="magic"):
        opened(b"DL4VCZR2" + blob[8:])
    with pytest.raises(ValueError, match="version"):
        opened(blob[:8] + np.uint32(2).tobytes() + blob[12:])
    ix = int(h["index_off"])
    for rec, (off, ln) in ((3, (int(h["data_bytes"]) - 10, 11)), (0, (2 ** 64 - 1, 1)), (4, (0, 2 ** 32 - 1))):
        entry = np.array([(off, ln)], dtype=[("o", "<u8"), ("l", "<u4")]).tobytes()
        with pytest.raises(ValueError, match=f"record {rec}"):
            opened(blob[:ix + 12 * rec] + entry + blob[ix + 12 * rec + 12:])
    assert len(opened(blob)) == 5


def test_zlib_device_decode_checks_buffers_before_any_device_work(synth_pair):
    """Staging or workspace too small returns DAN_E_WORKSPACE and an index entry outside the streams region DAN_E_INVALID, before
    the header pass, any copy or launch, so these run without a GPU."""
    from dl4vc_b200 import _lib
    from dl4vc_b200.feeder import _batch_struct, _decode_layout, _feeder_cfg, _scalars
    _, cf = synth_pair
    n, m = 3, cf.max_stream_bytes
    lay = _decode_layout(_lib.RECORDS_ZLIB, n, m)
    need = lay.staging_bytes
    staging = np.zeros(need, np.uint8)
    # the last stream ends at the end of the buffer, so the call needs the whole workspace
    staging[lay.stream_offsets:lay.stream_offsets + 8 * n].view(np.uint64)[:] = need - lay.streams - (n - np.arange(n)) * m
    staging[lay.stream_lengths:lay.stream_lengths + 4 * n].view(np.uint32)[:] = m
    sc = _scalars(n)
    out = _batch_struct([torch.zeros(1, dtype=torch.uint8) for _ in range(6)], sc)
    cfg, idx = _feeder_cfg(100, 200, 1, 1, 0, 0), np.arange(n, dtype=np.int64)
    ws, status = np.zeros(16, np.uint8), np.zeros(n, np.int32)
    lib = _lib.load_library()
    call = lambda sb, wb, c=cfg: lib.dan_decode_records_device(_lib.RECORDS_ZLIB, staging.ctypes.data, sb, idx.ctypes.data, n, C.byref(c),
                                                               C.byref(out), ws.ctypes.data, wb, status.ctypes.data, None)
    assert call(lay.streams - 1, lay.workspace_bytes) == -4 and b"staging buffer" in lib.dan_last_error()
    assert call(need, lay.workspace_bytes - 1) == -4 and b"device workspace" in lib.dan_last_error()
    assert call(need - 16, lay.workspace_bytes) == -1 and b"leaves the" in lib.dan_last_error()      # the last stream no longer fits
    assert call(need, lay.workspace_bytes, _feeder_cfg(201, 200, 1, 1, 0, 0)) == -1 and b"max_reads" in lib.dan_last_error()
    assert not sc["num_reads"].any(), "the header pass must not run before the checks"


# ---- GPU: inflate against zlib.decompress -------------------------------------------------------------------------------------------
class _BitWriter:
    """LSB-first DEFLATE bit writer for hand-made fixed-Huffman streams (zlib's encoder never emits some legal codes)."""

    def __init__(self):
        self.acc, self.n = 0, 0

    def bits(self, v, k):
        self.acc |= v << self.n
        self.n += k

    def huff(self, code, k):                   # Huffman codes go MSB first
        self.bits(int(format(code, f"0{k}b")[::-1], 2), k)

    def lit(self, s):
        if s < 144:
            self.huff(0x30 + s, 8)
        elif s < 256:
            self.huff(0x190 + s - 144, 9)
        elif s < 280:
            self.huff(s - 256, 7)
        else:
            self.huff(0xC0 + s - 280, 8)

    def match258(self, dist):
        self.lit(285)
        d = next(k for k in range(29, -1, -1) if (1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537,
                                                       2049, 3073, 4097, 6145, 8193, 12289, 16385, 24577)[k] <= dist)
        base = (1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097, 6145, 8193, 12289, 16385, 24577)[d]
        self.huff(d, 5)
        self.bits(dist - base, max(0, d // 2 - 1))


def fixed_stream(literals: bytes, matches: int, dist: int, payload_check=True) -> bytes:
    """zlib stream: one fixed-Huffman block of `literals`, then `matches` length-258 matches at distance `dist`."""
    w = _BitWriter()
    w.bits(1, 1); w.bits(1, 2)
    for b in literals:
        w.lit(b)
    for _ in range(matches):
        w.match258(dist)
    w.lit(256)
    body = w.acc.to_bytes((w.n + 7) // 8, "little")
    out = literals
    for _ in range(matches):
        for _ in range(258):
            out += out[len(out) - dist:len(out) - dist + 1]
    return b"\x78\x01" + body + zlib.adler32(out).to_bytes(4, "big")


def _inflate(streams, slot):
    from dl4vc_b200.feeder import inflate_device
    lens = [len(z) for z in streams]
    offs = np.concatenate(([0], np.cumsum(lens)[:-1])).astype(np.int64) + 3          # odd start: no alignment assumed
    src = torch.from_numpy(np.frombuffer(b"\xff" * 3 + b"".join(streams) + b"\xff" * 5, np.uint8).copy()).cuda()
    dst, st = inflate_device(src, torch.from_numpy(offs), torch.tensor(lens, dtype=torch.int32), slot)
    torch.cuda.synchronize()
    return dst.cpu().numpy(), st.cpu().numpy()


def _deflate(data, level=6, strategy=zlib.Z_DEFAULT_STRATEGY):
    c = zlib.compressobj(level, zlib.DEFLATED, 15, 9, strategy)
    return c.compress(data) + c.flush()


_SLOT = 40000


def _payloads():
    """name -> (zlib stream, data) for a _SLOT-byte payload of each kind the kernel must handle."""
    recs = make_records(4, seed=9, noise_rows=False)
    rec = _raw_bytes(recs)
    rng = np.random.default_rng(3)
    head = rng.integers(0, 256, 32768, dtype=np.uint8).tobytes()
    far = fixed_stream(head + head[:8], 28, 32768)
    out = {}
    for lv in (0, 1, 6, 9):
        out[f"level{lv}"] = rec[lv * 1000:lv * 1000 + _SLOT]
    for name, s in (("filtered", zlib.Z_FILTERED), ("huffman_only", zlib.Z_HUFFMAN_ONLY), ("rle", zlib.Z_RLE), ("fixed", zlib.Z_FIXED)):
        out[name] = (s, rec[70000:70000 + _SLOT])
    out["random"] = rng.integers(0, 256, _SLOT, dtype=np.uint8).tobytes()
    out["zeros"] = bytes(_SLOT)
    res = {}
    for k, v in out.items():
        if isinstance(v, tuple):
            res[k] = (_deflate(v[1], 6, v[0]), v[1])
        else:
            res[k] = (_deflate(v, int(k[5:]) if k.startswith("level") else 6), v)
    res["distance32768"] = (far, zlib.decompress(far))
    for z, d in res.values():
        assert zlib.decompress(z) == d and len(d) == _SLOT
    return res


@pytest.mark.gpu
def test_inflate_equals_zlib_on_every_block_kind():
    p = _payloads()
    names = list(p)
    for name in names:                                          # each kind alone
        dst, st = _inflate([p[name][0]], _SLOT)
        assert st.tolist() == [0], name
        assert dst[0].tobytes() == p[name][1], name
    order = [names[k % len(names)] for k in range(3 * len(names) + 1)]
    dst, st = _inflate([p[k][0] for k in order], _SLOT)        # one batch mixing all of them
    assert not st.any()
    for r, k in enumerate(order):
        assert dst[r].tobytes() == p[k][1], (r, k)


@pytest.mark.gpu
@pytest.mark.parametrize("level", [0, 1, 6, 9])
def test_inflate_equals_zlib_on_whole_records(level):
    recs = make_records(6, seed=12, depths=DEPTHS)
    recs[3:] = make_records(3, seed=13, noise_rows=False)
    streams = [_deflate(_raw_bytes(r), level) for r in recs] + [_deflate(_raw_bytes(recs[1]), level, s)
                                                                for s in (zlib.Z_FILTERED, zlib.Z_HUFFMAN_ONLY, zlib.Z_RLE, zlib.Z_FIXED)]
    dst, st = _inflate(streams, RECORD_BYTES)
    assert not st.any()
    for k, z in enumerate(streams):
        assert dst[k].tobytes() == zlib.decompress(z), k


@pytest.mark.gpu
@pytest.mark.parametrize("data", [b"", b"a", b"abcab", b"\x00" * 3, bytes(range(256))])
def test_inflate_equals_zlib_on_tiny_payloads(data):
    streams = [_deflate(data, lv) for lv in (0, 1, 9)] + [_deflate(data, 6, zlib.Z_FIXED)]
    dst, st = _inflate(streams, len(data))
    assert not st.any() and all(dst[k].tobytes() == data for k in range(len(streams)))


@pytest.mark.gpu
def test_inflate_rejects_invalid_streams_and_keeps_the_valid_ones():
    p = _payloads()
    good = [p[k][0] for k in ("level6", "random", "distance32768", "level0")]
    z = p["level6"][0]
    w = _BitWriter()                                            # dynamic block whose code-length code has 19 one-bit codes
    w.bits(1, 1); w.bits(2, 2); w.bits(0, 5); w.bits(0, 5); w.bits(15, 4)
    for _ in range(19):
        w.bits(1, 3)
    oversubscribed = b"\x78\x01" + w.acc.to_bytes((w.n + 7) // 8 + 8, "little")
    short_slot = _deflate(p["level6"][1][:-1])
    long_slot = _deflate(p["level6"][1] + b"x")
    bad = {
        "truncated": (z[:len(z) // 2], 5),
        "no_trailer": (z[:-4], 5),
        "adler": (z[:-1] + bytes([z[-1] ^ 1]), 8),
        "header": (b"\x78\x00" + z[2:], 1),
        "block_type3": (b"\x78\x01\x07" + bytes(16), 2),
        "stored_nlen": (b"\x78\x01\x01\x05\x00\x00\x00" + bytes(16), 2),
        "too_far": (fixed_stream(b"ab", 1, 3), 4),
        "code_set": (oversubscribed, 3),
        "longer": (long_slot, 6),
        "shorter": (short_slot, 7),
    }
    for name, (s, _) in bad.items():
        with pytest.raises(zlib.error) if name not in ("longer", "shorter") else contextlib.nullcontext():
            zlib.decompress(s)
    streams = []
    for k, (s, _) in enumerate(bad.values()):
        streams += [good[k % len(good)], s]
    dst, st = _inflate(streams, _SLOT)
    for k, (name, (s, code)) in enumerate(bad.items()):
        assert st[2 * k] == 0 and dst[2 * k].tobytes() == zlib.decompress(good[k % len(good)]), name
        assert st[2 * k + 1] == code, (name, int(st[2 * k + 1]))
        assert not dst[2 * k + 1].any(), name


# ---- GPU: compressed device decode == host decode of the raw records ----------------------------------------------------------------
def _assert_same_decode(rf, cf, idx, **kw):
    from dl4vc_b200.feeder import DeviceBatch, decode_records_device
    n = len(idx)
    R = kw.get("max_reads", 100)
    hb, sc_h = decode_records(rf, idx, HostBatch(max(n, 1), num_reads=R, pin=False), strict=False, **kw)
    db = DeviceBatch(n + 3, num_reads=R, max_stream_bytes=cf.max_stream_bytes)
    for t in (db.reads, db.q, db.strands, db.ref, db.ref_masks, db.var_masks):
        t.fill_(0xAB)
    db.inflate_status.fill_(-1)
    db, sc_d = decode_records_device(cf, idx, db, strict=False, **kw)
    torch.cuda.synchronize()
    for name, a, b in zip(("reads", "ref", "q", "strands", "ref_masks", "var_masks"), hb.tensors(), db.tensors()):
        assert tuple(a.shape) == tuple(b.shape), name
        assert np.array_equal(a.numpy(), b.cpu().numpy()), name
    for k in SCALAR_KEYS:
        assert np.array_equal(sc_h[k], sc_d[k]), k
    assert hb.meta == db.meta
    assert not db.inflate_status[:n].any()
    return sc_h


@pytest.mark.gpu
def test_compressed_device_decode_equals_host_decode_on_feeder_golden(tmp_path):
    recs = feeder_golden()["records"]
    path = str(tmp_path / "g.dz")
    write_compressed_records(path, recs.view(RECORD_DTYPE).reshape(-1), level=9)
    rf, cf = RecordFile(recs), CompressedRecordFile(path)
    n = len(rf)
    sc = _assert_same_decode(rf, cf, np.arange(n), seed=5)
    assert sc["status"].astype(bool).sum() == 3 and sc["blacklist"][1] == 1
    _assert_same_decode(rf, cf, np.random.default_rng(6).permutation(n), seed=6)


@pytest.mark.gpu
@pytest.mark.parametrize("kw", _CASES, ids=lambda k: "-".join(f"{a}{int(b)}" for a, b in k.items()))
def test_compressed_device_decode_equals_host_decode_on_synthetic_records(synth_pair, kw):
    rf, cf = synth_pair
    n = len(rf)
    sc = _assert_same_decode(rf, cf, np.arange(n), **kw)
    assert set(sc["num_reads"].tolist()) == set(DEPTHS) and (sc["status"] != 0).sum() == 2
    rng = np.random.default_rng(kw["seed"])
    _assert_same_decode(rf, cf, rng.choice(n, 37, replace=True), **kw)
    _assert_same_decode(rf, cf, np.arange(5, 18), **kw)
    _assert_same_decode(rf, cf, [n - 1], **kw)
    _assert_same_decode(rf, cf, np.zeros(0, np.int64), **kw)


@pytest.mark.gpu
def test_compressed_device_decode_by_path_and_argument_checks(synth_pair):
    from dl4vc_b200.feeder import DeviceBatch, decode_records_device
    rf, cf = synth_pair
    db, _ = decode_records_device(cf.path, np.arange(4), strict=False)
    torch.cuda.synchronize()
    assert db.max_stream_bytes == cf.max_stream_bytes and db.meta[3][0] == bytes(rf.field(3, "name")).decode()
    with pytest.raises(ValueError, match="max_stream_bytes"):
        decode_records_device(cf, np.arange(3), DeviceBatch(4))
    with pytest.raises(ValueError, match="max_stream_bytes"):
        decode_records_device(rf, np.arange(3), DeviceBatch(4, max_stream_bytes=100))
    with pytest.raises(ValueError, match="#7"):
        decode_records_device(cf, np.arange(9), DeviceBatch(9, max_stream_bytes=cf.max_stream_bytes))


# ---- GPU: call_record_file on a compressed file == on the raw file ------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("which", ["prod", "small"])
def test_call_record_file_compressed_equals_raw(which, tmp_path):
    from dl4vc_b200.config import prod_config, small_config
    from dl4vc_b200.factory import build_model
    from dl4vc_b200.feeder import REC_CORRUPT, call_record_file
    from dl4vc_b200.weights import synth_state_dict
    cfg = prod_config() if which == "prod" else small_config()
    model = build_model(cfg, synth_state_dict(cfg, seed=3), device="cuda:0").eval()
    n, broken = 300, (17, 18, 250)
    recs = make_records(n, seed=31, broken=broken)
    raw, cz = str(tmp_path / "r.bin"), str(tmp_path / "r.dz")
    recs.tofile(raw)
    write_compressed_records(cz, recs, level=1)
    thr = dict(snp=0.4, indel=0.2, long_indel=0.1)
    runs = [dict(batch_size=64), dict(batch_size=1036, depth=2), dict(batch_size=97, depth=1), dict(batch_size=64, depth=3),
            dict(start=40, stop=211, batch_size=50), dict(start=250, stop=251, batch_size=5)]
    for kw in runs:
        fr, fc = [], []
        want = _collect(call_record_file(model, raw, thresholds=thr, strict=False, failed=fr, **kw))
        got = _collect(call_record_file(model, cz, thresholds=thr, strict=False, failed=fc, **kw))
        assert got[0] == want[0] and got[1] == want[1], kw
        assert np.array_equal(got[2], want[2]) and np.array_equal(got[3], want[3]), kw
        assert fc == fr, kw
    clean = dict(start=19, stop=250, batch_size=100, thresholds=thr)
    a, b = _collect(call_record_file(model, raw, **clean)), _collect(call_record_file(model, CompressedRecordFile(cz), **clean))
    assert a[1] == b[1] and np.array_equal(a[2], b[2]) and np.array_equal(a[3], b[3])
    with pytest.raises(ValueError, match="#17"):
        _collect(call_record_file(model, cz, batch_size=64, thresholds=thr))

    # one corrupt stream: strict raises naming it when its batch finishes; non-strict reports it and keeps every other record
    cf = CompressedRecordFile(cz)
    bad_rec = 130
    blob = bytearray(open(cz, "rb").read())
    o = 64 + int(cf.offsets[bad_rec]) + int(cf.lengths[bad_rec]) // 2
    blob[o] ^= 0x5A
    corrupt = str(tmp_path / "corrupt.dz")
    with open(corrupt, "wb") as f:
        f.write(bytes(blob))
    with pytest.raises(ValueError, match=f"#{bad_rec}: compressed record is corrupt"):
        _collect(call_record_file(model, corrupt, start=100, stop=200, batch_size=16, thresholds=thr))
    fr, fc = [], []
    want = _collect(call_record_file(model, raw, batch_size=64, thresholds=thr, strict=False, failed=fr))
    got = _collect(call_record_file(model, corrupt, batch_size=64, thresholds=thr, strict=False, failed=fc))
    assert sorted(fc) == sorted(fr + [(bad_rec, REC_CORRUPT)])
    name = bytes(recs[bad_rec]["name"]).decode()
    keep = [k for k, nm in enumerate(want[0]) if nm != name]
    assert len(keep) == len(want[0]) - 1 and got[0] == [want[0][k] for k in keep] and got[1] == [want[1][k] for k in keep]
    assert np.array_equal(got[2], want[2][keep]) and np.array_equal(got[3], want[3][keep])
