"""GPU deflate (`dan_deflate_device`): every stream against zlib.decompress and the device inflate, the stored fallback and the size
bound, the window rules, determinism across batches and calls, the compressed size against zlib level 1, and compressed record files
written on the GPU against host-written ones."""
import ctypes as C
import os
import sys
import zlib

import numpy as np
import pytest
import torch

from test_gpu_compressed_records import _inflate, _raw_bytes
from test_gpu_record_calls import DEPTHS, _collect, feeder_golden, make_records
from dl4vc_b200.feeder import RECORD_BYTES, RECORD_DTYPE, CompressedRecordFile, RecordFile, write_compressed_records

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bound(s):
    return s + 5 * max(1, -(-s // 65535)) + 6


def _deflate_rows(rows):
    """rows: equal-length byte strings -> their GPU streams (bytes), after checking status, lengths and the packing."""
    from dl4vc_b200.feeder import deflate_device
    slot = len(rows[0]) if rows else RECORD_BYTES
    src = torch.from_numpy(np.frombuffer(b"".join(rows), np.uint8).copy().reshape(len(rows), slot)).cuda()
    streams, offsets, lengths, status = deflate_device(src)
    torch.cuda.synchronize()
    st, off, ln = status.cpu().numpy(), offsets.cpu().numpy(), lengths.cpu().numpy()
    assert not st.any()
    assert np.array_equal(off, np.concatenate(([0], np.cumsum(ln)[:-1])).astype(np.int64)) and streams.numel() == ln.sum()
    blob = streams.cpu().numpy().tobytes()
    return [blob[o:o + n] for o, n in zip(off, ln)]


def _check(rows):
    """Deflate rows on the GPU; each stream must fit the bound and inflate back exactly with zlib and with inflate_device."""
    streams = _deflate_rows(rows)
    for k, (z, r) in enumerate(zip(streams, rows)):
        assert len(z) <= _bound(len(r)), k
        assert zlib.decompress(z) == r, k
    if rows:
        dst, st = _inflate(streams, len(rows[0]))
        assert not st.any()
        for k, r in enumerate(rows):
            assert dst[k].tobytes() == r, k
    return streams


# ---- CPU: argument checks -------------------------------------------------------------------------------------------------------
def test_write_compressed_records_device_argument_checks(tmp_path):
    recs = make_records(2, seed=1, noise_rows=False)
    path = str(tmp_path / "r.dz")
    with pytest.raises(ValueError, match="level"):
        write_compressed_records(path, recs, level=6, device="cuda:0")
    with pytest.raises(ValueError, match="level and threads"):
        write_compressed_records(path, recs, threads=2, device="cuda:0")
    with pytest.raises(ValueError, match="CUDA device"):
        write_compressed_records(path, recs, device="cpu")


def test_deflate_device_argument_checks():
    from dl4vc_b200.feeder import deflate_device
    for bad in (torch.zeros((2, 8), dtype=torch.uint8), torch.zeros(8, dtype=torch.uint8), np.zeros((2, 8), np.uint8)):
        with pytest.raises(ValueError, match="CUDA uint8"):
            deflate_device(bad)


def test_deflate_entry_points_check_arguments_before_any_launch():
    """n < 0, null pointers and slots beyond the shared-memory capacity fail, and n = 0 succeeds, all without a launch, so these
    run without a GPU."""
    from dl4vc_b200 import _lib
    from dl4vc_b200.feeder import deflate_bound
    lib = _lib.load_library()
    for s in (0, 1, 258, 65535, 65536, 65537, RECORD_BYTES, 131072):
        assert deflate_bound(s) == _bound(s), s
    p = C.c_void_p(16)
    f = lib.dan_deflate_device
    assert f(p, -1, 100, p, p, p, None) == -1 and b"negative" in lib.dan_last_error()
    assert f(p, 3, 131073, p, p, p, None) == -2 and b"131072" in lib.dan_last_error()
    for args in ((None, 3, 100, p, p, p), (p, 3, 100, None, p, p), (p, 3, 100, p, None, p), (p, 3, 100, p, p, None)):
        assert f(*args, None) == -1 and b"null" in lib.dan_last_error(), args
    assert f(None, 0, 100, None, None, None, None) == 0
    assert lib.dan_deflate_compact(p, p, -1, 100, p, p, None) == -1
    assert lib.dan_deflate_compact(p, p, 2, 100, p, None, None) == -1


# ---- GPU: every stream inflates back -----------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_records_at_every_depth_round_trip():
    recs = make_records(2 * len(DEPTHS), seed=17, depths=DEPTHS, broken=(3, 12))
    clean = make_records(3, seed=18, noise_rows=False)
    golden = feeder_golden()["records"].view(RECORD_DTYPE).reshape(-1)
    rows = [_raw_bytes(r) for r in np.concatenate([recs, clean, golden])] + [bytes(RECORD_BYTES)]
    streams = _check(rows)
    assert len(streams[-1]) < 1000                                  # the all-zero record is long runs


@pytest.mark.gpu
def test_random_bytes_take_the_stored_fallback():
    rng = np.random.default_rng(5)
    rows = [rng.integers(0, 256, RECORD_BYTES, dtype=np.uint8).tobytes() for _ in range(3)]
    for z in _check(rows):
        assert len(z) == _bound(RECORD_BYTES)
        assert z[2] & 6 == 0                                        # BTYPE 00: stored


@pytest.mark.gpu
@pytest.mark.parametrize("size", [1, 2, 3, 4, 257, 258, 259, 65535, 65536, 65537])
def test_sizes_round_trip(size):
    rng = np.random.default_rng(size)
    rec = _raw_bytes(make_records(1, seed=size % 7, noise_rows=False))
    rows = [bytes(size), (b"abc" * size)[:size], rng.integers(0, 256, size, dtype=np.uint8).tobytes(),
            rng.integers(0, 4, size, dtype=np.uint8).tobytes(), (rec * 2)[:size]]
    streams = _check(rows)
    if size >= 65535:
        assert len(streams[0]) < size // 100 and len(streams[1]) < size // 100


@pytest.mark.gpu
@pytest.mark.parametrize("far", [32768, 32769])
def test_window_limit(far):
    """A random head followed by a copy of its start: the copy sits at distance `far`. 32768 is inside the window and compresses the
    copy; 32769 is not, so the copy stays literal and the stream cannot be much shorter than its input."""
    rng = np.random.default_rng(far)
    k = 4000
    head = rng.integers(0, 256, far, dtype=np.uint8).tobytes()
    data = head + head[:k]
    (z,) = _check([data])
    if far == 32768:
        assert len(z) < len(data) - k // 2, len(z)
    else:
        assert len(z) > len(data) - k // 8, len(z)


@pytest.mark.gpu
def test_runs_longer_than_258():
    parts = [b"A" * 1000, b"B" * 5000, b"ABAB" * 700, bytes(259), b"\xff" * 258, b"xy" * 129]
    data = b"".join(parts)
    (z,) = _check([data])
    assert len(z) < 300, len(z)


# ---- GPU: determinism -------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_stream_depends_only_on_its_input():
    recs = make_records(37, seed=23, depths=DEPTHS, broken=(4,))
    rows = [_raw_bytes(r) for r in recs]
    alone = [_deflate_rows([r])[0] for r in rows]
    batch = _deflate_rows(rows)
    assert batch == alone
    assert _deflate_rows(rows) == batch                            # a repeat call
    r = rows[9]
    assert _deflate_rows([r] * 37) == [alone[9]] * 37               # the same record at every position of a batch
    shuffled = np.random.default_rng(1).permutation(37)
    assert _deflate_rows([rows[k] for k in shuffled]) == [alone[k] for k in shuffled]


@pytest.mark.gpu
def test_empty_batch_succeeds():
    from dl4vc_b200.feeder import deflate_device
    streams, offsets, lengths, status = deflate_device(torch.zeros((0, RECORD_BYTES), dtype=torch.uint8, device="cuda"))
    assert streams.numel() == 0 and offsets.numel() == 0 and lengths.numel() == 0 and status.numel() == 0


# ---- GPU: size against zlib level 1 -------------------------------------------------------------------------------------------------
SIZE_BAR = 1.25                                                     # GPU stream bytes over zlib level 1's


def _bench_records(n, seed, tmp_path):
    sys.path.insert(0, os.path.join(ROOT, "scripts"))
    try:
        from bench_record_calls import write_records
    finally:
        sys.path.pop(0)
    path = str(tmp_path / "bench.bin")
    write_records(path, n, seed)
    return np.fromfile(path, dtype=RECORD_DTYPE)


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["make_records", "write_records"])
def test_size_against_zlib_level_1(which, tmp_path):
    recs = make_records(45, seed=21, depths=DEPTHS, broken=(7, 30)) if which == "make_records" else _bench_records(200, 2026, tmp_path)
    rows = [_raw_bytes(r) for r in recs]
    gpu = sum(len(z) for z in _check(rows))
    host = sum(len(zlib.compress(r, 1)) for r in rows)
    print(f"{which}: GPU {gpu / len(rows):.0f} B/record, zlib level 1 {host / len(rows):.0f} B/record, ratio {gpu / host:.3f}")
    assert gpu <= SIZE_BAR * host, gpu / host


# ---- GPU: compressed record files written on the GPU --------------------------------------------------------------------------------
@pytest.mark.gpu
def test_device_written_file_equals_host_written_file(tmp_path):
    recs = make_records(300, seed=31, depths=DEPTHS, broken=(17, 18, 250))
    dev_path, host_path = str(tmp_path / "d.dz"), str(tmp_path / "h.dz")
    slices = [recs[a:b] for a, b in ((0, 7), (7, 7), (7, 263), (263, 264), (264, 300))]    # growing, empty and one-record chunks
    assert write_compressed_records(dev_path, iter(slices), device="cuda:0") == len(recs)
    write_compressed_records(host_path, recs, level=1)
    cd, ch = CompressedRecordFile(dev_path), CompressedRecordFile(host_path)
    assert len(cd) == len(recs)
    cd.unpack(str(tmp_path / "d.bin"))
    with open(tmp_path / "d.bin", "rb") as f:
        assert f.read() == _raw_bytes(recs)
    assert np.array_equal(np.asarray(cd.sidecars), np.asarray(ch.sidecars))
    assert int(cd.lengths.astype(np.uint64).sum()) == len(cd.data)
    assert np.array_equal(cd.offsets, np.concatenate(([0], np.cumsum(cd.lengths.astype(np.uint64))[:-1])).astype(np.uint64))
    # the RecordFile source and the array source give the same file
    again = str(tmp_path / "d2.dz")
    write_compressed_records(again, RecordFile(recs), device=torch.device("cuda", 0))
    assert open(again, "rb").read() == open(dev_path, "rb").read()


@pytest.mark.gpu
def test_call_record_file_on_device_written_file_equals_raw(tmp_path):
    from dl4vc_b200.config import small_config
    from dl4vc_b200.factory import build_model
    from dl4vc_b200.feeder import call_record_file
    from dl4vc_b200.weights import synth_state_dict
    cfg = small_config()
    model = build_model(cfg, synth_state_dict(cfg, seed=3), device="cuda:0").eval()
    recs = make_records(300, seed=31, broken=(17, 18, 250))
    raw, cz = str(tmp_path / "r.bin"), str(tmp_path / "r.dz")
    recs.tofile(raw)
    write_compressed_records(cz, recs, device="cuda:0")
    thr = dict(snp=0.4, indel=0.2, long_indel=0.1)
    for kw in (dict(batch_size=64), dict(start=40, stop=211, batch_size=50, depth=3)):
        fr, fc = [], []
        want = _collect(call_record_file(model, raw, thresholds=thr, strict=False, failed=fr, **kw))
        got = _collect(call_record_file(model, cz, thresholds=thr, strict=False, failed=fc, **kw))
        assert got[0] == want[0] and got[1] == want[1], kw
        assert np.array_equal(got[2], want[2]) and np.array_equal(got[3], want[3]), kw
        assert fc == fr, kw
