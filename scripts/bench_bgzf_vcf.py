"""BGZF VCF output on one GPU: the BGZF deflate kernel alone, BgzfVcfWriter on the GPU against host zlib at levels 1 and 6, and
write_scored_vcf against call_record_file alone. Prints one JSON line with the GPU's name and power limit, read in the same run.

    python scripts/bench_bgzf_vcf.py [--kernel-mb 256] [--lines 400000] [--records 4144] [--batch 1036] [--out DIR]

Every timing ends in a device synchronise. The kernel runs on device-resident input larger than the 126 MB L2. Files go to a
temporary directory (or --out)."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HEADER = "##fileformat=VCFv4.2\n" + "".join(f"##contig=<ID=chr{c}>\n" for c in range(1, 23)) + \
    "#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\tSAMPLE\n"


def synthetic_scored_lines(n, seed, contigs=3):
    """n lines shaped like call_record_file's (the score field spliced into column 3), sorted, over `contigs` contigs."""
    rng = np.random.default_rng(seed)
    per = -(-n // contigs)
    bases = np.array(list("ACGT"))
    out = []
    for c in range(contigs):
        k = min(per, n - c * per)
        pos = 1000 + np.cumsum(rng.integers(1, 400, k))
        sc = rng.random((k, 4))
        ref_len = np.where(rng.random(k) < 0.85, 1, rng.integers(2, 12, k))
        for j in range(k):
            ref = "".join(bases[rng.integers(0, 4, ref_len[j])])
            alt = bases[rng.integers(0, 4)]
            out.append(f"chr{c + 1}\t{pos[j]}\tBP={sc[j, 0]:.8f};NV={sc[j, 1]:.8f};HV={sc[j, 2]:.8f};OV={sc[j, 3]:.8f}\t{ref}\t{alt}\t50\t.\t"
                       f"AF={sc[j, 1]:.4f};DP={int(sc[j, 2] * 90) + 5}\tGT\t0/1")
    return out


def _gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        name, power = [x.strip() for x in r.stdout.strip().splitlines()[0].split(",")]
        return name, power
    except Exception as e:                                       # the name still comes from torch
        import torch
        return torch.cuda.get_device_name(0), f"unknown ({e})"


def bench_kernel(mb, reps):
    import torch
    from dl4vc_b200.vcf import bgzf_compress_device
    text = ("\n".join(synthetic_scored_lines(40000, 7)) + "\n").encode()
    nbytes = mb << 20
    src = torch.from_numpy(np.frombuffer((text * (nbytes // len(text) + 1))[:nbytes], np.uint8).copy()).cuda()
    bgzf_compress_device(src[:1 << 20])                           # warm-up: module load, shared-memory attribute
    torch.cuda.synchronize()
    times, out = [], None
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = bgzf_compress_device(src)
        b.record()
        torch.cuda.synchronize()
        times.append(a.elapsed_time(b) / 1e3)
    t = min(times)
    blocks = len(out[2])
    return {"input_mb": mb, "blocks": blocks, "ms": round(t * 1e3, 2), "text_MB_per_s": round(nbytes / t / 1e6, 1),
            "blocks_per_s": round(blocks / t, 1), "ratio": round(int(out[0].numel()) / nbytes, 4)}


def _write(path, lines, batch, **kw):
    """-> (seconds to write and close, of which the index build, file bytes)"""
    from dl4vc_b200.vcf import BgzfVcfWriter
    t0 = time.perf_counter()
    with BgzfVcfWriter(path, HEADER, **kw) as w:
        for lo in range(0, len(lines), batch):
            w.write(lines[lo:lo + batch])
    return time.perf_counter() - t0, w.index_seconds, os.path.getsize(path)


def bench_writer(lines, batch, out):
    nbytes = sum(map(len, lines)) + len(lines)
    res = {"lines": len(lines), "text_MB": round(nbytes / 1e6, 2)}
    _write(os.path.join(out, "warm.vcf.gz"), lines[:20000], batch, device="cuda:0")
    for name, kw in (("gpu", dict(device="cuda:0")), ("host_zlib1", dict(level=1)), ("host_zlib6", dict(level=6))):
        t, t_index, size = _write(os.path.join(out, f"{name}.vcf.gz"), lines, batch, **kw)
        res[name] = {"s": round(t, 3), "lines_per_s": round(len(lines) / t), "MB_per_s": round(nbytes / t / 1e6, 1),
                     "bytes_per_line": round(size / len(lines), 2), "index_build_s": round(t_index, 3)}
    # host zlib level 6 alone, one thread: the compression cost per line the GPU path takes off the host
    import zlib
    text = ("\n".join(lines) + "\n").encode()
    t0 = time.perf_counter()
    for lo in range(0, len(text), 65280):
        c = zlib.compressobj(6, zlib.DEFLATED, -15)
        c.compress(text[lo:lo + 65280]); c.flush(); zlib.crc32(text[lo:lo + 65280])
    res["host_zlib6_us_per_line"] = round((time.perf_counter() - t0) / len(lines) * 1e6, 3)
    res["gpu_over_zlib1_bytes"] = round(res["gpu"]["bytes_per_line"] / res["host_zlib1"]["bytes_per_line"], 4)
    return res


def bench_scored(records, batch, out):
    import torch
    from bench_record_calls import write_records
    from dl4vc_b200.config import prod_config
    from dl4vc_b200.factory import build_model
    from dl4vc_b200.feeder import RecordFile, call_record_file, write_compressed_records
    from dl4vc_b200.vcf import write_scored_vcf
    from dl4vc_b200.weights import synth_state_dict
    cfg = prod_config()
    model = build_model(cfg, synth_state_dict(cfg, seed=1), device="cuda:0", precision="bf16").eval()
    raw, cz = os.path.join(out, "r.bin"), os.path.join(out, "r.dz")
    write_records(raw, records, 2026)
    write_compressed_records(cz, RecordFile(raw), device="cuda:0")
    for _ in call_record_file(model, cz, stop=batch, batch_size=batch):    # warm-up
        pass
    res = {}
    for rep in range(2):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        n = sum(len(l) for _, l, _, _ in call_record_file(model, cz, batch_size=batch, strict=False))
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        write_scored_vcf(os.path.join(out, "s.vcf.gz"), model, cz, HEADER, batch_size=batch, sort=True, strict=False)
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        res = {"records": records, "batch": batch, "lines": n, "call_record_file_us_per_record": round((t1 - t0) / records * 1e6, 2),
               "write_scored_vcf_us_per_record": round((t2 - t1) / records * 1e6, 2),
               "writer_us_per_record": round(((t2 - t1) - (t1 - t0)) / records * 1e6, 2)}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--kernel-mb", type=int, default=256)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--lines", type=int, default=400000)
    ap.add_argument("--batch-lines", type=int, default=1036)
    ap.add_argument("--records", type=int, default=4144)
    ap.add_argument("--batch", type=int, default=1036)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_bgzf_vcf.py needs a CUDA device")
    sys.path.insert(0, os.path.join(ROOT, "scripts"))
    name, power = _gpu_info()
    with tempfile.TemporaryDirectory() as tmp:
        out = a.out or tmp
        os.makedirs(out, exist_ok=True)
        res = {"gpu": name, "power_limit": power, "kernel": bench_kernel(a.kernel_mb, a.reps),
               "writer": bench_writer(synthetic_scored_lines(a.lines, 11), a.batch_lines, out),
               "scored_vcf": bench_scored(a.records, a.batch, out)}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
