"""Compressed record files against raw ones: size, host cost, H2D bytes, the inflate kernel and PROD bf16 file -> calls throughput.

One run writes the same seeded --records PROD-shaped records (bench_record_calls.write_records: 200 stored rows, num_reads uniform in
0..200) raw and compressed (write_compressed_records, zlib --level) into a temporary directory, reads both once so the page cache is
warm, and reports:
  * the compression ratio and bytes per record;
  * host microseconds per record of the device path's host work (staging copy + header pass + enqueue inside decode_records_device),
    compressed against raw, and the staging copy and the header pass (sidecars against raw records) alone;
  * H2D bytes per record of one staging copy, from the staging layout (dan_decode_layout) and the streams' lengths;
  * the inflate kernel alone (dan_inflate_device over one batch's streams already on the device): CUDA events around each launch,
    time per record and output GB/s, and, in a separate torch.profiler pass over the compressed device decode, the device time of
    inflate_kernel, decode_tiles_kernel and the H2D copy per record;
  * PROD bf16 records/s through call_record_file from the compressed file and from the raw file, alternated, over --passes passes;
  * the GPU's name and power limit.
Prints one JSON line (--out also writes it to a file).

    python scripts/bench_compressed_records.py --records 4144 --batch 1036 --passes 5
"""
from __future__ import annotations

import argparse
import json
import os
import shutil
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "scripts")):
    if p not in sys.path:
        sys.path.insert(0, p)


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--records", type=int, default=4144)
    ap.add_argument("--batch", type=int, default=1036, help="records per batch (1036 = 7 x 148)")
    ap.add_argument("--passes", type=int, default=5, help="timed passes over the file per measurement")
    ap.add_argument("--level", type=int, default=6, help="zlib level of the compressed file")
    ap.add_argument("--seed", type=int, default=2026)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if args.records < 1 or args.batch < 1 or args.passes < 1:
        ap.error("--records, --batch and --passes must be >= 1")

    import numpy as np
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_compressed_records.py measures on a CUDA device; none is visible")
    from bench_record_calls import power_limit_w, write_records
    from dl4vc_b200 import _lib
    from dl4vc_b200.config import prod_config
    from dl4vc_b200.factory import build_model
    from dl4vc_b200.feeder import (RECORD_BYTES, SIDECAR_BYTES, CompressedRecordFile, DeviceBatch, RecordFile, _decode_layout, _stage_streams,
                                   call_record_file, decode_record_headers, decode_records_device, inflate_device, write_compressed_records)
    from dl4vc_b200.weights import synth_state_dict

    dev = torch.device("cuda", 0)
    tmp = tempfile.mkdtemp(prefix="dl4vc_compressed_")
    try:
        raw_path, cz_path = os.path.join(tmp, "records.bin"), os.path.join(tmp, "records.dz")
        write_records(raw_path, args.records, args.seed)
        rf = RecordFile(raw_path)
        t0 = time.perf_counter()
        write_compressed_records(cz_path, rf, level=args.level)
        write_s = time.perf_counter() - t0
        cf = CompressedRecordFile(cz_path)
        N, B = len(rf), args.batch
        np.asarray(rf.raw).sum(dtype=np.uint64)
        np.asarray(cf.data).sum(dtype=np.uint64)
        starts = [(s, min(B, N - s)) for s in range(0, N, B)]
        cz_bytes = os.path.getsize(cz_path)
        result = {"device": torch.cuda.get_device_name(dev), "power_limit_w": power_limit_w(dev.index), "records": N, "batch": B,
                  "passes": args.passes, "zlib_level": args.level, "host_cpu": os.cpu_count(),
                  "file": {"raw_mb": round(N * RECORD_BYTES / 1e6, 1), "compressed_mb": round(cz_bytes / 1e6, 1),
                           "ratio": round(N * RECORD_BYTES / cz_bytes, 2), "compressed_bytes_per_record": round(cz_bytes / N, 1),
                           "stream_bytes_per_record": round(float(cf.lengths.mean()), 1), "max_stream_bytes": cf.max_stream_bytes,
                           "write_s": round(write_s, 2)},
                  "file_read": "np.memmap of files in a temporary directory, page cache warm (read once before timing)"}

        db_raw = DeviceBatch(B, device=dev)
        db_cz = DeviceBatch(B, device=dev, max_stream_bytes=cf.max_stream_bytes)

        def per_record_us(fn):
            best = float("inf")
            for _ in range(args.passes):
                t = 0.0
                for s, n in starts:
                    t0 = time.perf_counter()
                    fn(s, n)
                    t += time.perf_counter() - t0
                    torch.cuda.synchronize()
                best = min(best, t)
            return round(best / N * 1e6, 2)

        lay = lambda n: _decode_layout(_lib.RECORDS_ZLIB, n)

        def stage_compressed(s, n):
            st, L = db_cz.staging.numpy(), lay(n)
            st[L.sidecars:L.sidecars + n * SIDECAR_BYTES].reshape(n, SIDECAR_BYTES)[:] = cf.sidecars[s:s + n]
            _stage_streams(cf, np.arange(s, s + n), st[L.streams:])

        result["host_us_per_record"] = {
            "device_path_host_work_raw": per_record_us(lambda s, n: decode_records_device(rf, np.arange(s, s + n), db_raw, strict=False)),
            "device_path_host_work_compressed": per_record_us(lambda s, n: decode_records_device(cf, np.arange(s, s + n), db_cz, strict=False)),
            "staging_copy_raw": per_record_us(lambda s, n: rf.read_block(s, n, db_raw.staging)),
            "staging_copy_compressed": per_record_us(stage_compressed),
            "header_pass_raw": per_record_us(lambda s, n: decode_record_headers(rf, np.arange(s, s + n))),
            "header_pass_sidecar": per_record_us(lambda s, n: decode_record_headers(cf, np.arange(s, s + n))),
            "timing": "best of --passes passes, host clock around each call, device synchronised between calls"}
        copied = lambda L: L.streams - L.records         # the one H2D copy: from the records region to the streams, plus the used streams
        raw_h2d = sum(copied(_decode_layout(_lib.RECORDS_RAW, n)) for _, n in starts)
        cz_h2d = sum(copied(lay(n)) + int(cf.lengths[s:s + n].sum()) for s, n in starts)
        result["h2d_bytes_per_record"] = {"raw": round(raw_h2d / N, 1), "compressed": round(cz_h2d / N, 1), "ratio": round(raw_h2d / cz_h2d, 2)}

        # ---- the inflate kernel alone, on one batch's streams resident on the device ----
        s0, n0 = starts[0]
        host = np.zeros(int(cf.lengths[:n0].sum()) + 16, np.uint8)
        offs = _stage_streams(cf, np.arange(n0), host)
        src = torch.from_numpy(host).to(dev)
        off_t, len_t = torch.from_numpy(offs.astype(np.int64)), torch.from_numpy(cf.lengths[:n0].astype(np.int32))
        dst, st = inflate_device(src, off_t, len_t, RECORD_BYTES)
        torch.cuda.synchronize()
        assert not st.any() and np.array_equal(dst[:4].cpu().numpy(), rf.raw[:4]), "inflate_device disagrees with the file"
        ms = []
        reps = max(10, 2 * args.passes)
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); inflate_device(src, off_t, len_t, RECORD_BYTES); e1.record(); e1.synchronize()
            ms.append(e0.elapsed_time(e1))
        med = float(np.median(ms))
        result["inflate_kernel"] = {"batch_records": n0, "ms_per_batch_median": round(med, 3), "ms_per_batch_min": round(min(ms), 3),
                                    "us_per_record": round(med * 1e3 / n0, 3), "output_gb_per_s": round(n0 * RECORD_BYTES / (med * 1e6), 1),
                                    "input_gb_per_s": round(int(cf.lengths[:n0].sum()) / (med * 1e6), 2),
                                    "source": f"CUDA events around each of {reps} launches of dan_inflate_device (the binding's host-side "
                                              "bounds check runs before e0 is recorded and its launch is inside the events)"}
        del dst, st

        from torch.profiler import ProfilerActivity, profile
        for s, n in starts:
            decode_records_device(cf, np.arange(s, s + n), db_cz, strict=False)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(args.passes):
                for s, n in starts:
                    decode_records_device(cf, np.arange(s, s + n), db_cz, strict=False)
            torch.cuda.synchronize()
        split = {"inflate_kernel": 0.0, "decode_tiles_kernel": 0.0, "Memcpy HtoD": 0.0}
        for e in prof.key_averages():
            t = getattr(e, "device_time_total", None)
            t = e.cuda_time_total if t is None else t
            for k in split:
                if k in e.key:
                    split[k] += t
        recs = N * args.passes
        result["compressed_device_decode_us_per_record"] = {k.replace(" ", "_"): round(v / recs, 3) for k, v in split.items()}
        result["compressed_device_decode_us_per_record"]["source"] = "torch.profiler CUDA activities over --passes passes of decode_records_device"
        del prof

        # ---- PROD bf16 file -> calls, compressed against raw ----
        cfg = prod_config()
        model = build_model(cfg, synth_state_dict(cfg, seed=1), device=dev, precision="bf16").eval()

        def drive(f):
            k = 0
            for names, lines, gt, q in call_record_file(model, f, batch_size=B, depth=2, strict=False):
                k += len(lines)
            return k

        assert drive(rf) == drive(cf)
        t_raw, t_cz = [], []
        for _ in range(args.passes):
            torch.cuda.synchronize(); t0 = time.perf_counter(); drive(rf); t_raw.append(time.perf_counter() - t0)
            torch.cuda.synchronize(); t0 = time.perf_counter(); drive(cf); t_cz.append(time.perf_counter() - t0)
        r_rate, c_rate = N / float(np.median(t_raw)), N / float(np.median(t_cz))
        # the forward's share of a batch, for the inflate kernel's time to be read against
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        decode_records_device(rf, np.arange(s0, s0 + n0), db_raw, strict=False)
        torch.cuda.synchronize()
        fwd = []
        for _ in range(3):
            e0.record(); model.forward_heads(*db_raw.tensors()); e1.record(); e1.synchronize()
            fwd.append(e0.elapsed_time(e1))
        result["prod_bf16"] = {"raw_file_records_per_s": round(r_rate, 1), "compressed_file_records_per_s": round(c_rate, 1),
                               "compressed_over_raw": round(c_rate / r_rate, 3),
                               "forward_ms_per_batch": round(float(np.median(fwd)), 3),
                               "inflate_over_forward": round(med / float(np.median(fwd)), 4),
                               "call_record_file": "batch_size --batch, depth 2, strict=False; VCF lines and genotype calls out",
                               "timing": "median of --passes passes each, raw and compressed alternated, host clock ending in a device synchronise; "
                                         "forward_ms_per_batch: CUDA events around forward_heads on one decoded batch"}
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
