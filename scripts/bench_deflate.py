"""GPU deflate against host zlib on the same records, in the same run.

One run writes --records seeded PROD-shaped records (bench_record_calls.write_records: 200 stored rows, num_reads uniform in 0..200)
raw into a temporary directory, reads them once so the page cache is warm, and reports:
  * the deflate kernel alone (dan_deflate_device over one --batch of records already on the device): CUDA events around each of
    the repeated launches, records/s and input GB/s, and the stream bytes per record;
  * write_compressed_records(device=cuda:0) end to end from the raw file (H2D, deflate, compaction, D2H, sidecars, file writes),
    best of --passes, and write_compressed_records with host zlib at levels 1 and 6 on all host threads, best of --passes;
  * bytes per record of each file's streams, and the ratio of the GPU streams' bytes to level 1's;
  * the GPU's name and power limit, and the host's CPU count.
Prints one JSON line (--out also writes it to a file).

    python scripts/bench_deflate.py --records 4144
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
    ap.add_argument("--batch", type=int, default=1036, help="records per kernel launch in the kernel-only measurement (1036 = 7 x 148)")
    ap.add_argument("--passes", type=int, default=3, help="timed passes per end-to-end measurement")
    ap.add_argument("--launches", type=int, default=20, help="timed launches in the kernel-only measurement")
    ap.add_argument("--seed", type=int, default=2026)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if args.records < 1 or args.batch < 1 or args.passes < 1 or args.launches < 1:
        ap.error("--records, --batch, --passes and --launches must be >= 1")

    import numpy as np
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_deflate.py measures on a CUDA device; none is visible")
    from bench_record_calls import power_limit_w, write_records
    from dl4vc_b200.feeder import RECORD_BYTES, CompressedRecordFile, RecordFile, deflate_device, write_compressed_records

    dev = torch.device("cuda", 0)
    tmp = tempfile.mkdtemp(prefix="dl4vc_deflate_")
    try:
        raw_path = os.path.join(tmp, "records.bin")
        write_records(raw_path, args.records, args.seed)
        rf = RecordFile(raw_path)
        N = len(rf)
        np.asarray(rf.raw).sum(dtype=np.uint64)
        result = {"device": torch.cuda.get_device_name(dev), "power_limit_w": power_limit_w(dev.index), "records": N,
                  "record_bytes": RECORD_BYTES, "host_cpu": os.cpu_count(), "passes": args.passes}

        # ---- the kernel alone, records resident on the device ----
        B = min(args.batch, N)
        src = torch.from_numpy(np.array(rf.raw[:B])).to(dev)
        streams, offsets, lengths, status = deflate_device(src)
        assert not status.any().item(), "deflate failed"
        from dl4vc_b200 import _lib
        from dl4vc_b200.feeder import deflate_bound
        lib = _lib.load_library()
        bound = deflate_bound(RECORD_BYTES)
        slots = torch.empty(B * bound, dtype=torch.uint8, device=dev)
        ln, st = torch.empty(B, dtype=torch.int32, device=dev), torch.empty(B, dtype=torch.int32, device=dev)
        launch = lambda: lib.dan_deflate_device(src.data_ptr(), B, RECORD_BYTES, slots.data_ptr(), ln.data_ptr(), st.data_ptr(),
                                                torch.cuda.current_stream(dev).cuda_stream)
        for _ in range(3):
            assert launch() == 0
        torch.cuda.synchronize()
        ms = []
        for _ in range(args.launches):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); launch(); e1.record(); e1.synchronize()
            ms.append(e0.elapsed_time(e1))
        assert torch.equal(ln, lengths), "a repeated launch changed a stream length"
        med = float(np.median(ms))
        result["deflate_kernel"] = {"batch_records": B, "ms_per_batch_median": round(med, 3), "ms_per_batch_min": round(min(ms), 3),
                                    "records_per_s": round(B / (med * 1e-3), 1), "input_gb_per_s": round(B * RECORD_BYTES / (med * 1e6), 2),
                                    "stream_bytes_per_record": round(float(lengths.double().mean().item()), 1),
                                    "source": f"CUDA events around each of {args.launches} launches of dan_deflate_device after 3 warm-up "
                                              "launches; the input (B x 124 KB) stays in L2 between launches"}
        del src, streams, offsets, slots

        # ---- end to end: raw file -> compressed record file ----
        def best_write(path, **kw):
            best = float("inf")
            for _ in range(args.passes):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                write_compressed_records(path, rf, **kw)
                best = min(best, time.perf_counter() - t0)
            cf = CompressedRecordFile(path)
            return {"records_per_s": round(N / best, 1), "s": round(best, 3),
                    "stream_bytes_per_record": round(float(cf.lengths.astype(np.float64).mean()), 1),
                    "file_bytes_per_record": round(os.path.getsize(path) / N, 1)}

        gpu_path, l1_path, l6_path = (os.path.join(tmp, f) for f in ("gpu.dz", "l1.dz", "l6.dz"))
        e2e = {"gpu": best_write(gpu_path, device=dev), "host_zlib_level1": best_write(l1_path, level=1),
               "host_zlib_level6": best_write(l6_path, level=6)}
        e2e["host_threads"] = min(32, os.cpu_count() or 1)
        e2e["gpu_bytes_over_level1"] = round(e2e["gpu"]["stream_bytes_per_record"] / e2e["host_zlib_level1"]["stream_bytes_per_record"], 3)
        e2e["timing"] = "best of --passes passes of write_compressed_records from the raw file (page cache warm) to a file in a temporary directory"
        result["write_compressed_records"] = e2e
        check = CompressedRecordFile(gpu_path).records([0, N - 1])
        assert check.tobytes() == np.ascontiguousarray(rf.raw[[0, N - 1]]).tobytes(), "the GPU-written file does not inflate to the records"
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
