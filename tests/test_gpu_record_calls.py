"""Record file -> scored VCF records and genotype calls: the header pass of the decode (CPU), the device tile pass
(`dan_decode_records_device`, byte-for-byte against the host decode) and the streaming driver `call_record_file` against the manual
composition decode_records -> forward_heads_host -> scores_on_device -> genotype_calls_on_device -> splice_vcf_records."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN_DIR
from dl4vc_b200.feeder import (RECORD_BYTES, RECORD_DTYPE, HostBatch, RecordFile, decode_record_headers, decode_records)
from dl4vc_b200.synth import make_pileups

LETTER = {1: "A", 2: "T", 3: "G", 4: "C", 5: "-"}
DEPTHS = (0, 1, 37, 99, 100, 101, 150, 200)
SCALAR_KEYS = ("label", "num_reads", "is_snp", "var_type", "allele_freq", "coverage", "var_base_enum", "var_ref_enum", "blacklist", "status")


def make_records(n, seed, depths=None, noise_rows=True, broken=()):
    """n records of RECORD_DTYPE around synthetic pileups of up to 200 stored rows. depths: num_reads of each record (cycled);
    noise_rows: stored rows past the pileup hold random tokens, so a wrong row pick shows; broken: records whose VCF line the
    reference's loader raises on (equal-length non-SNP alleles)."""
    rng = np.random.default_rng(seed + 1)
    rec = np.zeros(n, dtype=RECORD_DTYPE)
    for lo in range(0, n, 128):
        hi = min(n, lo + 128)
        b = make_pileups(hi - lo, seed=seed * 7919 + lo, num_reads=200, coverage="ragged", max_depth=200)
        for k in range(hi - lo):
            i = lo + k
            d = int(b.num_reads[k])
            rec[i]["name"] = f"chr{1 + i % 22}:{1000 + i}".encode()
            rec[i]["single_reads"] = b.reads[k].T
            rec[i]["q-scores"] = b.q_scores[k].T
            rec[i]["strand"] = b.strands[k].T
            if noise_rows and d < 200:
                rec[i]["single_reads"][d:] = rng.integers(1, 10, (200 - d, 201))
                rec[i]["q-scores"][d:] = rng.integers(2, 42, (200 - d, 201))
                rec[i]["strand"][d:] = rng.integers(1, 3, (200 - d, 201))
            rec[i]["ref_bases"] = b.ref[k]
            rec[i]["num_reads"] = d if depths is None else depths[i % len(depths)]
            rec[i]["label"] = i % 3
            rm, vm = b.ref_masks[k], b.var_masks[k]
            nz = np.flatnonzero(rm)
            if b.kind[k] == 0:
                x, y = LETTER[int(rm[100])], LETTER[int(vm[100])]
            elif b.kind[k] == 1:
                x, y = LETTER[int(rm[100])], "".join(LETTER[int(v)] for v in vm[nz])
            else:
                x, y = "".join(LETTER[int(v)] for v in rm[nz]), LETTER[int(vm[100])]
            if i in broken:
                x, y = "AT", "GC"
            gt = ["", "\tGT:0/1", "\tGT:1/1"][i % 3]
            rec[i]["vcfrec"] = f"chr{1 + i % 22}\t{1000 + i}\t.\t{x}\t{y}\t50\t.\tAF={rng.random():.4f};DP={int(rng.integers(5, 90))}\tGT\t0/1{gt}".encode()
    return rec


def feeder_golden():
    return np.load(os.path.join(GOLDEN_DIR, "feeder.npz"))


# ---- CPU: header pass, record blocks, argument checks ----------------------------------------------------------------------------
@pytest.mark.parametrize("max_reads,store,seed", [(100, 200, 5), (20, 50, 6), (200, 200, 1), (1, 100, 2)])
def test_header_pass_names_the_host_tile_columns(max_reads, store, seed):
    g = feeder_golden()
    recs = np.concatenate([g["records"].view(RECORD_DTYPE).reshape(-1), make_records(24, seed=11, depths=DEPTHS)])
    rf = RecordFile(recs)
    n = len(rf)
    idx = np.arange(n)
    kw = dict(seed=seed, max_reads=max_reads, store_max_reads=store)
    hdr, sc_h, rm, vm = decode_record_headers(rf, idx, **kw)
    batch, sc = decode_records(rf, idx, HostBatch(n, num_reads=max_reads, pin=False), strict=False, **kw)
    for k in SCALAR_KEYS:
        assert np.array_equal(sc_h[k], sc[k]), k
    assert np.array_equal(rm, batch.ref_masks.numpy()) and np.array_equal(vm, batch.var_masks.numpy())
    tiles = (batch.reads.numpy(), batch.q.numpy(), batch.strands.numpy())
    for i in range(n):
        h = hdr[i]
        m = int(h["num_rows"])
        rows = h["rows"][:m].astype(np.int64)
        S = min(store, 200)
        assert 0 <= m <= max_reads and np.all(np.diff(rows) > 0)
        assert np.all(rows >= h["window_start"]) and np.all(rows < min(200, int(h["window_start"]) + S))
        for t, name in zip(tiles, ("single_reads", "q-scores", "strand")):
            assert np.array_equal(t[i][:, :m], recs[i][name][rows].T), (i, name)
            assert not t[i][:, m:].any(), (i, name)
        fields = bytes(recs[i]["vcfrec"]).decode().strip().split("\t")
        if len(fields) >= 8:
            assert (h["ref_len"], h["var_len"]) == (len(fields[3]), len(fields[4]))


def test_record_blocks_read_and_gather_raw_bytes():
    rf = RecordFile(make_records(9, seed=3, noise_rows=False))
    out = np.zeros(10 * RECORD_BYTES, np.uint8)
    rf.read_block(2, 5, out)
    assert np.array_equal(out[:5 * RECORD_BYTES], rf.raw[2:7].reshape(-1)) and not out[5 * RECORD_BYTES:].any()
    rf.gather([8, 0, 8, 3], torch.from_numpy(out))
    assert np.array_equal(out[:4 * RECORD_BYTES].reshape(4, -1), rf.raw[[8, 0, 8, 3]])
    with pytest.raises(IndexError):
        rf.read_block(6, 4, out)
    with pytest.raises(IndexError):
        rf.gather([9], out)
    with pytest.raises(ValueError, match="need"):
        rf.read_block(0, 9, np.zeros(3 * RECORD_BYTES, np.uint8))


def test_raw_device_decode_rejects_bad_arguments_before_any_device_work():
    """Out-of-range indices raise in Python; a staging buffer or workspace below the size the call needs returns DAN_E_WORKSPACE
    before any copy or launch, so both checks run without a GPU."""
    from dl4vc_b200 import _lib
    from dl4vc_b200.feeder import _batch_struct, _decode_layout, _feeder_cfg, _scalars, decode_records_device
    rf = RecordFile(make_records(3, seed=4, noise_rows=False))
    with pytest.raises(IndexError, match="out of range"):
        decode_records_device(rf, [0, 3])
    with pytest.raises(IndexError, match="out of range"):
        decode_records_device(rf, [-1])
    lib = _lib.load_library()
    n = 3
    lay = _decode_layout(_lib.RECORDS_RAW, n)
    need = lay.staging_bytes
    assert need >= n * RECORD_BYTES + n * (216 + 2 * 201)
    staging = np.zeros(need, np.uint8)
    staging[lay.records:lay.records + n * RECORD_BYTES] = rf.raw.reshape(-1)
    tiles = [torch.zeros(1, dtype=torch.uint8) for _ in range(6)]
    sc = _scalars(n)
    out = _batch_struct(tiles, sc)
    cfg = _feeder_cfg(100, 200, 1, 1, 0, 0)
    idx = np.arange(n, dtype=np.int64)
    ws = np.zeros(16, np.uint8)
    call = lambda c, sb, wb: lib.dan_decode_records_device(_lib.RECORDS_RAW, staging.ctypes.data, sb, idx.ctypes.data, n, C.byref(c), C.byref(out),
                                                           ws.ctypes.data, wb, None, None)
    assert call(cfg, need - 1, lay.workspace_bytes) == -4 and b"staging buffer" in lib.dan_last_error()
    assert call(cfg, need, lay.workspace_bytes - 1) == -4 and b"device workspace" in lib.dan_last_error()
    assert not sc["num_reads"].any(), "the header pass must not run before the size checks"
    assert call(_feeder_cfg(201, 200, 1, 1, 0, 0), need, lay.workspace_bytes) == -1 and b"max_reads" in lib.dan_last_error()


@pytest.mark.parametrize("n", [0, 1, 3, 1036])
def test_decode_layout_regions(n):
    """dan_decode_layout for both formats: each region 16-byte aligned, disjoint, inside the staging buffer, the streams last; the
    sidecars before the copied range [records, streams + used streams); the copy carries the records (raw) or the index (compressed),
    the headers and the masks, and besides them only alignment padding: the parent's packing, which left the two mask regions
    unaligned, copied at most 32 bytes less, and exactly as many for the 1036-record batches of the benchmarks."""
    from dl4vc_b200 import _lib
    from dl4vc_b200.feeder import SIDECAR_BYTES, _decode_layout
    a16 = lambda x: -(-x // 16) * 16
    m = 1000
    for fmt in (_lib.RECORDS_RAW, _lib.RECORDS_ZLIB):
        z = fmt == _lib.RECORDS_ZLIB
        lay = _decode_layout(fmt, n, m)
        sizes = {"sidecars": z * n * SIDECAR_BYTES, "records": (not z) * n * RECORD_BYTES, "stream_offsets": z * 8 * n,
                 "stream_lengths": z * 4 * n, "headers": 216 * n, "ref_masks": 201 * n, "var_masks": 201 * n, "streams": z * n * m}
        spans = sorted((getattr(lay, k), getattr(lay, k) + v, k) for k, v in sizes.items())
        assert all(lo % 16 == 0 for lo, _, _ in spans), spans
        assert all(hi <= nxt for (_, hi, _), (nxt, _, _) in zip(spans, spans[1:])), spans
        assert spans[-1][1] <= lay.staging_bytes and lay.streams >= max(hi for _, hi, k in spans if k != "streams")
        assert lay.sidecars + sizes["sidecars"] <= lay.records
        copied = [k for lo, hi, k in spans if lay.records <= lo and hi <= lay.streams and hi > lo]
        assert copied == ([] if n == 0 else ["stream_offsets", "stream_lengths"] if z else ["records"]) + (["headers", "ref_masks", "var_masks"] if n else [])
        copy = lay.streams - lay.records
        index = a16(n * SIDECAR_BYTES)
        before = a16(a16(index + 12 * n) + 618 * n) - index if z else a16(a16(n * RECORD_BYTES) + 618 * n)
        assert before <= copy <= before + 32 and (n != 1036 or copy == before), (copy, before)
        assert lay.workspace_bytes == (a16(n * RECORD_BYTES) if z else 0) + lay.staging_bytes - lay.records


# ---- GPU: device decode == host decode, byte for byte ----------------------------------------------------------------------------
def _assert_same_decode(rf, idx, **kw):
    from dl4vc_b200.feeder import DeviceBatch, decode_records_device
    n = len(idx)
    R = kw.get("max_reads", 100)
    hb, sc_h = decode_records(rf, idx, HostBatch(max(n, 1), num_reads=R, pin=False), strict=False, **kw)
    db = DeviceBatch(n + 3, num_reads=R)
    for t in (db.reads, db.q, db.strands, db.ref, db.ref_masks, db.var_masks):
        t.fill_(0xAB)                      # every output byte must be written
    db, sc_d = decode_records_device(rf, idx, db, strict=False, **kw)
    torch.cuda.synchronize()
    for name, a, b in zip(("reads", "ref", "q", "strands", "ref_masks", "var_masks"), hb.tensors(), db.tensors()):
        assert tuple(a.shape) == tuple(b.shape), name
        assert np.array_equal(a.numpy(), b.cpu().numpy()), name
    for k in SCALAR_KEYS:
        assert np.array_equal(sc_h[k], sc_d[k]), k
    assert hb.meta == db.meta
    return sc_h


@pytest.mark.gpu
@pytest.mark.parametrize("seed", [5, 6])
def test_device_decode_equals_host_decode_on_feeder_golden(seed):
    rf = RecordFile(feeder_golden()["records"])
    n = len(rf)
    sc = _assert_same_decode(rf, np.arange(n), seed=seed)
    assert sc["status"].astype(bool).sum() == 3 and sc["blacklist"][1] == 1
    _assert_same_decode(rf, np.random.default_rng(seed).permutation(n), seed=seed)


_CASES = [dict(max_reads=100, store_max_reads=200, seed=0), dict(max_reads=100, store_max_reads=100, seed=1),
          dict(max_reads=20, store_max_reads=50, seed=0), dict(max_reads=200, store_max_reads=200, seed=1),
          dict(max_reads=1, store_max_reads=200, seed=0), dict(max_reads=100, store_max_reads=50, seed=1, use_q_scores=False),
          dict(max_reads=200, store_max_reads=100, seed=0, use_strands=False),
          dict(max_reads=20, store_max_reads=200, seed=1, use_q_scores=False, use_strands=False, keep_candidate_af=True)]


@pytest.fixture(scope="module")
def synth_file():
    return RecordFile(make_records(45, seed=21, depths=DEPTHS, broken=(7, 30)))


@pytest.mark.gpu
@pytest.mark.parametrize("kw", _CASES, ids=lambda k: "-".join(f"{a}{int(b)}" for a, b in k.items()))
def test_device_decode_equals_host_decode_on_synthetic_records(synth_file, kw):
    rf = synth_file
    n = len(rf)
    sc = _assert_same_decode(rf, np.arange(n), **kw)                             # read_block path, 45 records
    assert set(sc["num_reads"].tolist()) == set(DEPTHS) and (sc["status"] != 0).sum() == 2
    rng = np.random.default_rng(kw["seed"])
    _assert_same_decode(rf, rng.choice(n, 37, replace=True), **kw)               # shuffled, repeated: gather path
    _assert_same_decode(rf, np.arange(5, 18), **kw)                              # a sub-range: the draw keys on the file index
    _assert_same_decode(rf, [n - 1], **kw)
    _assert_same_decode(rf, np.zeros(0, np.int64), **kw)


@pytest.mark.gpu
def test_device_decode_argument_checks_raise_before_launch():
    from dl4vc_b200.feeder import DeviceBatch, decode_records_device
    rf = RecordFile(make_records(6, seed=8, noise_rows=False))
    db = DeviceBatch(4)
    db.reads.fill_(7)
    with pytest.raises(ValueError, match="capacity"):
        decode_records_device(rf, np.arange(6), db)
    with pytest.raises(ValueError, match="max_reads"):
        decode_records_device(rf, np.arange(3), db, max_reads=50)
    with pytest.raises(IndexError):
        decode_records_device(rf, [0, 6], db)
    torch.cuda.synchronize()
    assert bool((db.reads == 7).all())
    bad = RecordFile(make_records(6, seed=8, noise_rows=False, broken=(2,)))
    with pytest.raises(ValueError, match="#2"):
        decode_records_device(bad, np.arange(4), db)


# ---- GPU: the streaming driver against the manual composition --------------------------------------------------------------------
def _manual_calls(model, rf, idx, thresholds):
    from dl4vc_b200.feeder import genotype_calls_on_device, scores_on_device, splice_vcf_records
    hb, _ = decode_records(rf, idx, HostBatch(len(idx), num_reads=model.num_single_reads), use_q_scores=model.use_q_scores,
                           use_strands=model.use_strands, max_reads=model.num_single_reads)
    heads = model.forward_heads_host(*hb.tensors())
    torch.cuda.synchronize()
    scores = scores_on_device(heads.cuda())
    fields = [v.strip().split("\t") for _, v in hb.meta]
    rl = torch.tensor([len(f[3]) for f in fields], dtype=torch.int32)
    vl = torch.tensor([len(f[4]) for f in fields], dtype=torch.int32)
    gt, q = genotype_calls_on_device(scores, rl, vl, **thresholds)
    s = scores.cpu().numpy()
    lines = splice_vcf_records([v for _, v in hb.meta], s[:, 0], s[:, 1:])
    return [m for m, _ in hb.meta], lines, gt.cpu().numpy(), q.cpu().numpy(), heads.clone()


def _collect(gen):
    names, lines, gts, qs = [], [], [], []
    for a, b, c, d in gen:
        assert len(a) == len(b) == len(c) == len(d)
        names += a; lines += b; gts.append(c); qs.append(d)
    return names, lines, np.concatenate(gts) if gts else np.zeros(0, np.int8), np.concatenate(qs) if qs else np.zeros(0, np.int32)


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["prod", "small"])
def test_call_record_file_equals_manual_composition(which, tmp_path):
    from dl4vc_b200.config import prod_config, small_config
    from dl4vc_b200.factory import build_model
    from dl4vc_b200.feeder import DeviceBatch, call_record_file, decode_records_device
    from dl4vc_b200.weights import synth_state_dict
    cfg = prod_config() if which == "prod" else small_config()
    model = build_model(cfg, synth_state_dict(cfg, seed=3), device="cuda:0").eval()
    n, broken = 300, (17, 18, 250)
    path = str(tmp_path / "records.bin")
    make_records(n, seed=31, broken=broken).tofile(path)
    rf = RecordFile(path)
    good = np.array([i for i in range(n) if i not in broken])
    thr = dict(snp=0.4, indel=0.2, long_indel=0.1)
    names, lines, gt, q, heads = _manual_calls(model, rf, good, thr)
    assert (gt > 0).any() and (gt == 0).any()

    # the heads themselves: the device decode feeds forward_heads the same bytes
    db, _ = decode_records_device(rf, good, DeviceBatch(len(good), model.num_single_reads), max_reads=model.num_single_reads,
                                  use_q_scores=model.use_q_scores, use_strands=model.use_strands)
    assert torch.equal(model.forward_heads(*db.tensors()).cpu(), heads)

    failed = []
    got = _collect(call_record_file(model, path, batch_size=64, thresholds=thr, strict=False, failed=failed))
    assert got[0] == names and got[1] == lines
    assert np.array_equal(got[2], gt) and np.array_equal(got[3], q)
    assert sorted(i for i, _ in failed) == list(broken) and all(s == 3 for _, s in failed)
    for bs, depth in ((1036, 2), (97, 1), (64, 3)):
        again = _collect(call_record_file(model, rf, batch_size=bs, depth=depth, thresholds=thr, strict=False))
        assert again[1] == lines and np.array_equal(again[2], gt) and np.array_equal(again[3], q), (bs, depth)
    lo, hi = 40, 211
    sub = _collect(call_record_file(model, rf, start=lo, stop=hi, batch_size=50, thresholds=thr, strict=False))
    rows = np.flatnonzero((good >= lo) & (good < hi))
    assert sub[1] == [lines[r] for r in rows] and np.array_equal(sub[2], gt[rows]) and np.array_equal(sub[3], q[rows])
    clean = _collect(call_record_file(model, rf, start=19, stop=250, batch_size=100, thresholds=thr))
    assert clean[1] == [lines[r] for r in np.flatnonzero((good >= 19) & (good < 250))]
    with pytest.raises(ValueError, match="#17"):
        _collect(call_record_file(model, rf, batch_size=64, thresholds=thr))
