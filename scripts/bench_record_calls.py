"""Record file -> calls on the GPU: host cost of the decode and PROD bf16 throughput of call_record_file.

One run builds a seeded file of --records PROD-shaped records (200 stored rows each, num_reads uniform in 0..200; 4144 records are
514 MB, more than the 126 MB L2) in a temporary directory, reads it once so the page cache is warm, and reports:
  * host microseconds per record: the full host decode (dan_decode_records into a pinned HostBatch) against the host work of the
    device path (read_block + header pass + enqueue inside decode_records_device), and each of read_block and the header pass alone;
  * device time per record of the device decode: CUDA events around each call (staging H2D copy + tile kernel, both on one stream),
    and, in a separate torch.profiler pass with CUDA activities, the split into decode_tiles_kernel and the copy;
  * PROD bf16 records/s through call_record_file from the file, next to forward_heads_host on pre-decoded pinned tensors of the
    same records (the bench.py e2e input path), both over --passes passes after one warm-up pass;
  * the GPU's name and power limit.
Prints one JSON line (--out also writes it to a file).

    python scripts/bench_record_calls.py --records 4144 --batch 1036 --passes 5
"""
from __future__ import annotations

import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def power_limit_w(index: int = 0):
    try:
        import pynvml
        pynvml.nvmlInit()
        return pynvml.nvmlDeviceGetPowerManagementLimit(pynvml.nvmlDeviceGetHandleByIndex(index)) / 1000.0
    except Exception:
        pass
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return float(out)
    except Exception:
        return None


def write_records(path, n, seed):
    """n records of RECORD_DTYPE: synthetic pileups (dl4vc_b200.synth) with SNP / insert / delete VCF lines, num_reads 0..200."""
    import numpy as np
    from dl4vc_b200.feeder import RECORD_DTYPE
    from dl4vc_b200.synth import make_pileups
    letter = {1: "A", 2: "T", 3: "G", 4: "C", 5: "-"}
    rng = np.random.default_rng(seed)
    with open(path, "wb") as f:
        for lo in range(0, n, 128):
            m = min(n, lo + 128) - lo
            b = make_pileups(m, seed=seed + lo, num_reads=200, coverage="ragged", max_depth=200)
            rec = np.zeros(m, dtype=RECORD_DTYPE)
            rec["single_reads"] = b.reads.transpose(0, 2, 1)
            rec["q-scores"] = b.q_scores.transpose(0, 2, 1)
            rec["strand"] = b.strands.transpose(0, 2, 1)
            rec["ref_bases"] = b.ref
            rec["num_reads"] = rng.integers(0, 201, m)
            for k in range(m):
                i = lo + k
                rm, vm, nz = b.ref_masks[k], b.var_masks[k], np.flatnonzero(b.ref_masks[k])
                if b.kind[k] == 0:
                    x, y = letter[int(rm[100])], letter[int(vm[100])]
                elif b.kind[k] == 1:
                    x, y = letter[int(rm[100])], "".join(letter[int(v)] for v in vm[nz])
                else:
                    x, y = "".join(letter[int(v)] for v in rm[nz]), letter[int(vm[100])]
                rec[k]["name"] = f"chr{1 + i % 22}:{1000 + i}".encode()
                rec[k]["label"] = i % 3
                rec[k]["vcfrec"] = f"chr{1 + i % 22}\t{1000 + i}\t.\t{x}\t{y}\t50\t.\tAF={rng.random():.4f};DP={int(rng.integers(5, 90))}\tGT\t0/1".encode()
            rec.tofile(f)


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--records", type=int, default=4144)
    ap.add_argument("--batch", type=int, default=1036, help="records per batch (1036 = 7 x 148)")
    ap.add_argument("--passes", type=int, default=5, help="timed passes over the file per measurement")
    ap.add_argument("--seed", type=int, default=2026)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if args.records < 1 or args.batch < 1 or args.passes < 1:
        ap.error("--records, --batch and --passes must be >= 1")

    import numpy as np
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_record_calls.py measures on a CUDA device; none is visible")
    from dl4vc_b200 import _lib
    from dl4vc_b200.config import prod_config
    from dl4vc_b200.factory import build_model
    from dl4vc_b200.feeder import (RECORD_BYTES, DeviceBatch, HostBatch, RecordFile, _decode_layout, call_record_file, decode_record_headers,
                                   decode_records, decode_records_device)
    from dl4vc_b200.weights import synth_state_dict

    dev = torch.device("cuda", 0)
    tmp = tempfile.mkdtemp(prefix="dl4vc_records_")
    try:
        path = os.path.join(tmp, "records.bin")
        write_records(path, args.records, args.seed)
        rf = RecordFile(path)
        N, B = len(rf), args.batch
        np.asarray(rf.raw).sum(dtype=np.uint64)           # page cache warm
        starts = [(s, min(B, N - s)) for s in range(0, N, B)]
        result = {"device": torch.cuda.get_device_name(dev), "power_limit_w": power_limit_w(dev.index), "records": N,
                  "file_mb": round(N * RECORD_BYTES / 1e6, 1), "batch": B, "passes": args.passes,
                  "file_read": "np.memmap of a file in a temporary directory, page cache warm (read once before timing)",
                  "host_cpu": os.cpu_count()}

        # ---- host microseconds per record ----
        hb = HostBatch(B, pin=True)
        db = DeviceBatch(B, device=dev)
        stage = db.staging.numpy()[_decode_layout(_lib.RECORDS_RAW, B).records:]

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

        full = per_record_us(lambda s, n: decode_records(rf, np.arange(s, s + n), hb, strict=False))
        device_host = per_record_us(lambda s, n: decode_records_device(rf, np.arange(s, s + n), db, strict=False))
        read = per_record_us(lambda s, n: rf.read_block(s, n, stage))
        header = per_record_us(lambda s, n: decode_record_headers(rf, np.arange(s, s + n)))
        result["host_us_per_record"] = {"full_host_decode": full, "device_path_host_work": device_host, "read_block": read,
                                        "header_pass": header, "ratio_device_path_to_full": round(device_host / full, 3),
                                        "timing": "best of --passes passes, host clock around each call, device synchronised between calls"}

        # ---- device time of the tile pass ----
        from torch.profiler import ProfilerActivity, profile
        for s, n in starts:
            decode_records_device(rf, np.arange(s, s + n), db, strict=False)
        torch.cuda.synchronize()
        ev_ms = 0.0
        for _ in range(args.passes):
            for s, n in starts:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda._sleep(100_000_000)      # ~50 ms of device time: e0 then fires after the host pass has queued the copy
                e0.record()
                decode_records_device(rf, np.arange(s, s + n), db, strict=False)
                e1.record()
                e1.synchronize()
                ev_ms += e0.elapsed_time(e1)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(args.passes):
                for s, n in starts:
                    decode_records_device(rf, np.arange(s, s + n), db, strict=False)
            torch.cuda.synchronize()
        kern = copy = 0.0
        kcount = 0
        for e in prof.key_averages():
            name = e.key
            t = getattr(e, "device_time_total", None)
            t = e.cuda_time_total if t is None else t
            if "decode_tiles_kernel" in name:
                kern += t; kcount += e.count
            elif "Memcpy HtoD" in name:
                copy += t
        recs = N * args.passes
        layouts = [_decode_layout(_lib.RECORDS_RAW, n) for _, n in starts]
        h2d_bytes = args.passes * sum(L.streams - L.records for L in layouts)      # the one H2D copy of each call
        result["device_tile_pass"] = {"copy_plus_kernel_us_per_record_events": round(ev_ms * 1e3 / recs, 3),
                                      "kernel_us_per_record": round(kern / recs, 4), "launches": kcount,
                                      "staging_h2d_us_per_record": round(copy / recs, 3),
                                      "h2d_gb_per_s": round(h2d_bytes / (copy * 1e3), 1) if copy else None,
                                      "source": "copy_plus_kernel: CUDA events recorded around each call on its stream; kernel / copy split: "
                                                "torch.profiler CUDA activities over --passes further passes"}
        del prof

        # ---- PROD bf16: records/s from the file vs from pre-decoded pinned tensors ----
        cfg = prod_config()
        model = build_model(cfg, synth_state_dict(cfg, seed=1), device=dev, precision="bf16").eval()

        def drive():
            k = 0
            for names, lines, gt, q in call_record_file(model, rf, batch_size=B, depth=2, strict=False):
                k += len(lines)
            return k

        pre = []
        for s, n in starts:
            h, _ = decode_records(rf, np.arange(s, s + n), HostBatch(n, pin=True), strict=False)
            pre.append(h)
        outs = [torch.empty((h.size, 27), dtype=torch.float32).pin_memory() for h in pre]

        def pinned():
            for h, o in zip(pre, outs):
                model.forward_heads_host(*h.tensors(), out=o)
            torch.cuda.synchronize()

        drive(); pinned()
        t_file, t_pin = [], []
        for _ in range(args.passes):            # alternate the two, so both see the same clocks
            torch.cuda.synchronize(); t0 = time.perf_counter(); got = drive(); t_file.append(time.perf_counter() - t0)
            torch.cuda.synchronize(); t0 = time.perf_counter(); pinned(); t_pin.append(time.perf_counter() - t0)
        f_rate, p_rate = N / float(np.median(t_file)), N / float(np.median(t_pin))
        result["prod_bf16"] = {"call_record_file_records_per_s": round(f_rate, 1), "pinned_forward_heads_host_candidates_per_s": round(p_rate, 1),
                               "file_over_pinned": round(f_rate / p_rate, 3), "lines_per_pass": got,
                               "call_record_file": "read_block -> header pass -> H2D + tile pass (side stream) -> forward_heads -> dan_scores -> "
                                                   "dan_genotype_calls -> 16 B scores + gt/q D2H -> dan_format_vcf_info -> VCF lines, depth 2",
                               "pinned": "forward_heads_host on HostBatch tensors decoded before timing (heads D2H, no scoring, no VCF text)",
                               "timing": "median of --passes passes, host clock, each ending in a device synchronise"}
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
