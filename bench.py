#!/usr/bin/env python
"""bench.py — candidates/s of the DAN forward (BASELINE.json metric) on N B200s, one process per GPU.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--precision bf16|fp32] [--batch B] [--dump-outputs DIR]

A "step" is one pass of the hot path (encoder -> conv stack -> pooling -> FC -> heads, dl4vc/model.py:434-961) over one
batch of B synthetic PROD-shaped pileup candidates (100 reads x 201 positions, all read rows populated = the dense
worst case). Candidates are independent, so N GPUs shard by candidate with no collective ("scaling": "weak").

  value     whole-job candidates/s, inputs already resident in HBM (device pointers -> dan_forward)
  e2e       the same metric through the host-buffer call: pinned uint8 host tensors -> H2D -> dan_forward -> D2H of the
            (B,27) head matrix, every step, all inside the timed region
  roofline  dominant kernel class (conv stack) timed with CUDA events on the launching stream by the library's
            profile hook; tensor-pipe bound (SURVEY §8d: 2.65e5 FLOP/B >> ridge), peak = MEASURED_PEAKS.json
  cpu_baseline / --impl reference
            the reference's own torch-CPU op sequence (oracle/dan_torch_cpu.py — the reference is pure PyTorch and
            /root/reference does not exist on the GPU box) on all host cores, bounded sample of the same workload

The per-step batch (default 4144 candidates = 252 MB of uint8 input) is larger than the 126 MB L2, so no L2 flush is
needed between timed iterations.

--dump-outputs DIR writes the (B,27) fp32 head matrix of the last timed `value` step to DIR/heads.npy (DIR/heads_rank<r>.npy
per rank under torchrun). Inputs and weights are seeded, so two builds run with the same arguments can be compared output for
output. The dump stays within 64 MB in all: a rank's head matrix above 64 MB / N (N ranks) is cut to a fixed, seeded sample of its
rows (the same rows in every run of that batch size and rank count).

--steps K times K steps in every region that times this project's code (value, e2e, the profile pass, the fp32 and train blocks);
the CPU and torch-eager samples of the reference op sequence are baselines of fixed size.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "candidate variants/sec (DAN forward)"
UNIT = "candidates/s"
WORKLOAD = "PROD DAN forward (call_variants.sh:101-147 flag set: 7 conv layers x128ch, highway 32, FC 73856-1024-256), "\
           "100 reads x 201 bp, dense pileups, 1M-candidate job processed in per-step batches"


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return {"bf16_burst": float(d["bf16_tflops"]), "bf16_sustained": float(d.get("bf16_tflops_sustained", d["bf16_tflops"])),
                "hbm_gbs": float(d["hbm_gbs"]), "source": "measured"}
    return {"bf16_burst": 1590.0, "bf16_sustained": 1400.0, "hbm_gbs": 6650.0, "source": "fallback"}


def stack_kernel_traffic():
    """DRAM bytes (read + write) of the conv-stack kernel per launch and per candidate, from the committed `ncu --set full` capture of a
    148-candidate pass (profiles/r02_stack_kernel_ncu_full_summary.csv: one column per segment launch)."""
    import csv
    path = os.path.join(ROOT, "profiles", "r02_stack_kernel_ncu_full_summary.csv")
    if not os.path.exists(path):
        return None
    scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    total, launches, cands = 0.0, 0, 148
    with open(path) as f:
        for row in csv.reader(f):
            if row and row[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                vals = [float(v) * scale[row[1]] for v in row[2:] if v]
                total += sum(vals); launches = len(vals)
    if not launches:
        return None
    return {"per_launch": total / launches, "per_candidate": total / cands, "source": "ncu --set full, profiles/r02_stack_kernel_ncu_full_summary.csv"}


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons with NVML while the timed region runs."""

    def __init__(self, index: int, period_s: float = 0.1):
        super().__init__(daemon=True)
        self.index, self.period = index, period_s
        self.samples, self.reasons, self.power = [], set(), []
        self.max_mhz = None
        self._halt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception as e:  # NVML unavailable: record why
            self.err = repr(e)

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake",
        }
        while not self._halt.is_set():
            try:
                self.samples.append(int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                try:
                    self.power.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
                except Exception:
                    pass
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._halt.wait(self.period)

    def stop(self):
        self._halt.set()
        if self.is_alive():
            self.join(timeout=2)
        s = sorted(self.samples)
        med = s[len(s) // 2] if s else None
        pw = sorted(self.power)
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(s),
                "power_w": round(pw[len(pw) // 2], 1) if pw else None}


# ---------------------------------------------------------------------------------------------------------
def cpu_reference_rate(cfg, sd, sample, batch, repeats, warmup=1):
    """candidates/s of the reference's torch-CPU op sequence on this host (all cores)."""
    import torch

    from oracle import dan_torch_cpu

    torch.set_num_threads(os.cpu_count() or 1)
    arrs = sample.slice(0, batch).arrays()
    r, q, s, ref, rm, vm = arrs
    for _ in range(warmup):
        dan_torch_cpu.forward(cfg, sd, r, ref, q, s, rm, vm)
    times = []
    for _ in range(repeats):
        t0 = time.perf_counter()
        dan_torch_cpu.forward(cfg, sd, r, ref, q, s, rm, vm)
        times.append(time.perf_counter() - t0)
    return batch * len(times) / sum(times), times


def torch_eager_gpu_rate(cfg, sd, sample, dev, batch=16, repeats=10, warmup=4):
    """Second stated baseline (SURVEY section 2.1): the reference's own op sequence (oracle/dan_torch_cpu.py) as torch eager kernels on this
    GPU, fp32 with TF32 off — what running the reference's model.py on a B200 costs. A bounded sample; reported, not a target."""
    import torch

    from oracle import dan_torch_cpu

    tf32 = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    try:
        sd_dev = {k: (v.to(dev) if hasattr(v, "to") else torch.as_tensor(v).to(dev)) for k, v in sd.items()}
        r, q, s, ref, rm, vm = [torch.from_numpy(a).to(dev) for a in sample.slice(0, batch).arrays()]
        for _ in range(warmup):          # the GPU has idled through the CPU baseline: library initialisation and the clock ramp stay outside
            dan_torch_cpu.forward(cfg, sd_dev, r, ref, q, s, rm, vm)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(repeats):
            dan_torch_cpu.forward(cfg, sd_dev, r, ref, q, s, rm, vm)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        return {"value": batch * repeats / (ms * 1e-3), "unit": UNIT, "kind": "reference op sequence as torch eager CUDA kernels (cuDNN / cuBLAS fp32, TF32 off)",
                "sample": f"{repeats} timed batches x {batch} of the same dense PROD candidates ({warmup} warm-up), torch {torch.__version__}"}
    except Exception as exc:      # an out-of-memory or library failure of the baseline must not take the bench line down
        return {"value": None, "error": f"{type(exc).__name__}: {str(exc)[:160]}"}
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = tf32
        torch.cuda.empty_cache()


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import torch

    from dl4vc_b200.config import prod_config
    from dl4vc_b200.synth import make_pileups
    from dl4vc_b200.weights import synth_state_dict

    cfg = prod_config()
    sd = synth_state_dict(cfg, seed=1)
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    sample = make_pileups(256, seed=20261018, coverage="full")
    # size a step so that the whole run stays within a few minutes: probe 16 candidates, aim at ~2 s per step
    rate_probe, _ = cpu_reference_rate(cfg, sd, sample, 16, 1, warmup=1)
    per_step = int(min(256, max(16, (rate_probe * 2.0) // 16 * 16)))
    total_steps = args.steps + args.warmup
    while per_step > 16 and per_step * total_steps / rate_probe > 240:
        per_step -= 16
    from oracle import dan_torch_cpu

    r, q, s, ref, rm, vm = sample.slice(0, per_step).arrays()
    for _ in range(args.warmup):
        dan_torch_cpu.forward(cfg, sd, r, ref, q, s, rm, vm)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        dan_torch_cpu.forward(cfg, sd, r, ref, q, s, rm, vm)
    dt = time.perf_counter() - t0
    value = per_step * args.steps / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "candidates_per_step": per_step, "model": "PROD", "reads": cfg.num_reads, "window": cfg.read_len},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{args.steps} timed steps x {per_step} dense PROD candidates, torch {torch.__version__} CPU ops "
                                   "(oracle/dan_torch_cpu.py = the reference's own op sequence, fp32)"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


# ---------------------------------------------------------------------------------------------------------
def fma_peak_tflops(clocks):
    """fp32 FMA peak of this GPU: the nominal figure (148 SMs x 128 lanes x 2 x max SM clock) is the denominator; the rate a register-resident
    FFMA loop sustains (dan_measure_fma_tflops, ~40 ms on every SM — it runs into the power limit, the GEMM kernels do not) is reported beside it."""
    from dl4vc_b200 import _lib
    nominal = 148 * 128 * 2 * (clocks.get("sm_max_mhz") or 1965) * 1e6 / 1e12
    src = "nominal: 148 SMs x 128 FMA lanes x 2 x sm_max_mhz"
    try:
        import torch
        v = float(_lib.load_library().dan_measure_fma_tflops(40.0, torch.cuda.current_stream().cuda_stream))
        if v > 0:
            src += f"; a pure FFMA loop sustains {v:.1f} TFLOP/s on this GPU (dan_measure_fma_tflops, power-limited)"
    except Exception:
        pass
    return nominal, src


def fp32_block(model, sample, dev, cfg, clocks, batch=592, steps=3):
    """BASELINE configs[1]: the fp32 path (logits within 1e-4 of the reference, tests/test_gpu_parity.py) on 4 full passes, resident and
    through the host-buffer call. CUDA-core FFMA: quoted against the FMA peak of the part at the sampled maximum SM clock."""
    import numpy as np
    import torch
    from dl4vc_b200 import _lib
    reps = (batch + len(sample) - 1) // len(sample)
    host = [torch.from_numpy(np.ascontiguousarray(np.concatenate([a] * reps, axis=0)[:batch])).pin_memory() for a in sample.arrays()]
    h_r, h_q, h_s, h_ref, h_rm, h_vm = host
    d_r, d_q, d_s, d_ref, d_rm, d_vm = [t.to(dev) for t in host]
    model.set_precision("fp32")
    out_host = torch.empty((batch, _lib.NUM_HEAD_OUTPUTS), dtype=torch.float32).pin_memory()
    res = {}
    for name, fn in (("value", lambda: model.forward_heads(d_r, d_ref, d_q, d_s, d_rm, d_vm)),
                     ("e2e", lambda: model.forward_heads_host(h_r, h_ref, h_q, h_s, h_rm, h_vm, out=out_host))):
        for _ in range(2):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        res[name] = batch * steps / (e0.elapsed_time(e1) * 1e-3)
    model.set_precision("bf16")
    fma_peak, fma_src = fma_peak_tflops(clocks)
    ach = res["value"] * 2 * cfg.macs_per_candidate() / 1e12
    return {"value": res["value"], "e2e": res["e2e"], "unit": UNIT, "candidates_per_step": batch, "steps": steps, "dtype": "f32",
            "tolerance": "logits within 1e-4 relative of the reference (tests/test_gpu_parity.py)",
            "roofline": {"bound": "fp32_fma (CUDA cores)", "achieved": ach, "peak": fma_peak, "unit": "TFLOP/s", "frac": ach / fma_peak,
                         "peak_source": fma_src}}


def train_step_block(cfg, sd, dev, dist, world, rank, timed, batch=32, steps=3, e2e=False):
    """BASELINE configs[4]: one data-parallel training step per rank = training-mode forward (batch-statistics BatchNorm, dropout 0.1, read
    removal) -> device loss block (dan_losses) -> native backward -> bucketed gradient all-reduce over NCCL -> grad clip 1.0 -> Adam, with the
    close-example flags scattered into the device-resident table (easy-example down-sampling input). fp32 kernels; `value` counts the
    candidates of all ranks."""
    import numpy as np
    import torch
    from dl4vc_b200.factory import build_model
    from dl4vc_b200.losses import fused_losses, update_close_table
    from dl4vc_b200.synth import make_pileups
    from dl4vc_b200.train_dp import GradientAllReducer
    model = build_model(cfg, sd, device=dev, precision="fp32").train()
    opt = torch.optim.Adam(model.parameters(), lr=2e-4)            # main.py:116, train_variant_caller.sh
    reducer = GradientAllReducer(model)
    b = make_pileups(batch, seed=4242 + rank, coverage="poisson")
    d = [torch.from_numpy(np.ascontiguousarray(a)).to(dev) for a in b.arrays()]
    vt = torch.from_numpy(np.rint(b.var_fraction * 2).astype(np.int64)).to(dev)
    tb = (vt > 0).long()
    af = torch.from_numpy(b.var_fraction.astype(np.float32)).to(dev)
    cov = torch.from_numpy((b.num_reads * 0.01).astype(np.float32)).to(dev)
    vb = torch.from_numpy(b.var_masks[:, 100].astype(np.int64)).to(dev); vr = torch.from_numpy(b.ref_masks[:, 100].astype(np.int64)).to(dev)
    table = torch.zeros(1 << 20, dtype=torch.uint8, device=dev)
    idx = torch.arange(batch, device=dev) + rank * batch
    state = {}

    def step():
        opt.zero_grad(set_to_none=True)
        heads = model.forward_train_heads(d[0], d[3], d[1], d[2], d[4], d[5], rm_non_var_reads=0, rm_var_reads=1)
        total, comps, close_vt, _ = fused_losses(heads, tb, vt, af, cov, vb, vr)
        total.backward()
        reducer()
        torch.nn.utils.clip_grad_norm_(model.parameters(), 1.0)        # train_variant_caller.sh:104
        opt.step()
        update_close_table(table, idx, close_vt)
        state["loss"] = comps

    for _ in range(2):
        step()
    ms = timed(step, steps)
    launches = getattr(model, "last_train_launch_count", 0) + 2          # + dan_losses_kernel, close_table_update_kernel
    extra = {}
    if e2e:
        # the step a trainer runs per batch: pinned host uint8 tensors + labels -> device, the step, the loss block back to the host
        host = [torch.from_numpy(np.ascontiguousarray(a)).pin_memory() for a in b.arrays()]
        lab_host = [t.cpu().pin_memory() for t in (tb, vt, af, cov, vb, vr)]
        loss_host = torch.empty(8, dtype=torch.float32).pin_memory()

        def step_e2e():
            nonlocal d, tb, vt, af, cov, vb, vr
            d = [t.to(dev, non_blocking=True) for t in host]
            tb, vt, af, cov, vb, vr = [t.to(dev, non_blocking=True) for t in lab_host]
            step()
            loss_host.copy_(state["loss"].reshape(-1)[:8], non_blocking=True)

        step_e2e()
        ms_e2e = timed(step_e2e, steps)
        extra = {"e2e_ms": ms_e2e, "h2d_bytes_per_step": sum(t.numel() * t.element_size() for t in host + lab_host), "d2h_bytes_per_step": 32,
                 "launches_per_step": launches}
    grad_bytes = sum(p.numel() for p in model.parameters() if p.requires_grad) * 4
    loss = [round(float(x), 4) for x in state["loss"].cpu()]
    del model, opt
    torch.cuda.empty_cache()
    return {**extra, "value": batch * world * steps / (ms * 1e-3), "unit": "candidates/s (training step)", "batch_per_gpu": batch, "steps": steps, "ms_per_step": ms / steps,
            "dtype": "f32", "collective": None if world == 1 else f"NCCL all-reduce (sum / {world}) of {grad_bytes / 1e6:.0f} MB fp32 gradients per step in 2 buckets "
                                                                    "(FC trunk + heads first, on a side stream), BatchNorm statistics per GPU",
            "step": "train forward + dan_losses + dan_backward + gradient all-reduce + clip_grad_norm 1.0 + Adam + close-table scatter",
            "last_losses[bin,vt,af,cov,vb,vr,total,n_close]": loss}


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, name, arr, limit=DUMP_LIMIT_BYTES):
    """arr (rows x cols float32, host) -> out_dir/<name>.npy, above `limit` bytes a seeded row sample in ascending row order."""
    import numpy as np
    if arr.nbytes > limit:
        keep = limit // (arr.shape[1] * arr.itemsize)
        arr = arr[np.sort(np.random.default_rng(0).choice(arr.shape[0], keep, replace=False))]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(arr, dtype=np.float32))


def run_b200(args):
    import numpy as np
    import torch

    from dl4vc_b200 import _lib
    from dl4vc_b200.config import prod_config
    from dl4vc_b200.factory import build_model
    from dl4vc_b200.synth import make_pileups
    from dl4vc_b200.weights import synth_state_dict

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (the DAN forward has no CPU path)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # stdout carries the ONE JSON line only: NCCL prints its version banner (and, at NCCL_DEBUG=INFO, its log) to fd 1 when the
        # communicator is created, so fd 1 points at stderr until the first collective has run
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            warm = torch.zeros(1, device=dev)
            dist.all_reduce(warm)
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)

    lib = _lib.load_library()     # fails loudly if the CUDA library is missing
    cfg = prod_config()
    sd = synth_state_dict(cfg, seed=1)
    model = build_model(cfg, sd, device=dev, precision=args.precision)
    if args.pass_candidates:
        model.set_pass_candidates(args.pass_candidates)

    # ---- synthetic inputs: `unique` distinct candidates per rank, tiled to the step batch ---------------
    B = args.batch
    unique = min(B, 512)
    sample = make_pileups(unique, seed=20261018 + rank, coverage="full")
    reps = (B + unique - 1) // unique
    host = [torch.from_numpy(np.ascontiguousarray(np.concatenate([a] * reps, axis=0)[:B])).pin_memory() for a in sample.arrays()]
    h_r, h_q, h_s, h_ref, h_rm, h_vm = host
    d_r, d_q, d_s, d_ref, d_rm, d_vm = [t.to(dev) for t in host]
    in_bytes = sum(t.numel() for t in host)
    out_host = torch.empty((B, _lib.NUM_HEAD_OUTPUTS), dtype=torch.float32).pin_memory()

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if dist is not None:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        barrier()
        return ms

    if args.mode == "train":
        # BASELINE configs[4] as a line of its own: python bench.py --mode train [--gpus N under torchrun]
        sampler = ClockSampler(local)
        sampler.start()
        tb = train_step_block(cfg, sd, dev, dist, world, rank, timed, batch=args.train_batch, steps=args.steps, e2e=True)
        clocks = sampler.stop()
        if rank == 0:
            n = args.train_batch * world * args.steps
            print(json.dumps({
                "metric": "candidate variants/sec (DAN training step)", "value": tb["value"], "unit": "candidates/s", "n_gpus": world, "steps": args.steps,
                "warmup": 2, "ms_per_step": tb["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic", "mode": "train",
                "config": {"workload": "PROD DAN training step (train_variant_caller.sh flag set): " + tb["step"], "candidates_per_step_per_gpu": args.train_batch,
                           "model": "PROD", "parallelism": f"data-parallel x{world}", "collective": tb["collective"],
                           "l2_policy": "activation tape of a step (GBs) exceeds the 126 MB L2, no flush"},
                "e2e": {"value": n / (tb["e2e_ms"] * 1e-3), "unit": "candidates/s", "h2d_bytes_per_step": tb["h2d_bytes_per_step"],
                        "d2h_bytes_per_step": tb["d2h_bytes_per_step"], "ms_per_step": tb["e2e_ms"] / args.steps},
                "gpu_launches": tb["launches_per_step"] * args.steps, "clocks": clocks,
                "last_losses[bin,vt,af,cov,vb,vr,total,n_close]": tb["last_losses[bin,vt,af,cov,vb,vr,total,n_close]"]}), flush=True)
        if dist is not None:
            dist.destroy_process_group()
        return 0

    last = {}

    def step_resident():
        last["heads"] = model.forward_heads(d_r, d_ref, d_q, d_s, d_rm, d_vm)
        return last["heads"]

    def step_e2e():
        # pinned host uint8 -> chunked H2D on the library's side stream, overlapped with the kernels -> D2H of the (B,27) result
        return model.forward_heads_host(h_r, h_ref, h_q, h_s, h_rm, h_vm, out=out_host)

    # ---- warm-up, then the timed regions ------------------------------------------------------------------
    for _ in range(max(args.warmup, 3)):
        step_resident()
    sampler = ClockSampler(local)
    sampler.start()
    ms = timed(step_resident, args.steps)
    launches = model.last_launch_count * args.steps
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, "heads" if world == 1 else f"heads_rank{rank}", last["heads"].cpu().numpy(), DUMP_LIMIT_BYTES // world)
    for _ in range(2):
        step_e2e()
    ms_e2e = timed(step_e2e, args.steps)
    # dominant-kernel timing: the same steps with the library's event hook on
    lib.dan_profile_enable(1)
    prof_steps = args.steps
    timed(step_resident, prof_steps)
    import ctypes as C
    ms_cls = (C.c_double * _lib.PROF_NUM_CLASSES)()
    n_cls = (C.c_int * _lib.PROF_NUM_CLASSES)()
    _lib.check(lib.dan_profile_read(ms_cls, n_cls, _lib.PROF_NUM_CLASSES), "dan_profile_read")
    lib.dan_profile_enable(0)
    clocks = sampler.stop()

    train_block = None if args.no_train else train_step_block(cfg, sd, dev, dist, world, rank, timed, steps=args.steps)
    total_cands = B * world * args.steps
    value = total_cands / (ms * 1e-3)
    e2e_value = total_cands / (ms_e2e * 1e-3)
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return 0

    peaks = load_peaks()
    traffic = stack_kernel_traffic()
    R, P, Cc = cfg.num_reads, cfg.read_len, cfg.channels
    # conv-stack class = conv(1x3) + residual 1x1 + bottleneck 1x1 MACs (SURVEY App. E); compression/FC/heads run in the GEMM class
    macs_conv_stack = 0
    cin = cfg.in_channels
    for l in range(1, cfg.total_conv_layers + 1):
        macs_conv_stack += R * P * Cc * cin * 3
        cin = Cc
        if cfg.is_residual(l):
            macs_conv_stack += R * P * Cc * Cc
        if cfg.highway:
            macs_conv_stack += R * P * Cc * cfg.bottleneck
    flops_total = 2 * cfg.macs_per_candidate()
    cls_names = [lib.dan_profile_class_name(i).decode() for i in range(_lib.PROF_NUM_CLASSES)]
    cls_ms = {cls_names[i]: ms_cls[i] / prof_steps for i in range(_lib.PROF_NUM_CLASSES)}
    cls_n = {cls_names[i]: n_cls[i] // prof_steps for i in range(_lib.PROF_NUM_CLASSES)}
    dom = "conv_stack"
    dom_ms_step = cls_ms[dom]
    dom_launches = max(cls_n[dom], 1)
    flops_per_launch = 2.0 * macs_conv_stack * B / dom_launches
    achieved = flops_per_launch / (dom_ms_step / dom_launches * 1e-3) / 1e12 if dom_ms_step > 0 else 0.0
    peak = peaks["bf16_sustained"] if args.precision == "bf16" else None
    roofline = {
        "bound": "tensor", "kernel": "dan_stack_kernel (conv stack class)", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
        "frac": (achieved / peak) if peak else None,
        # dram__bytes_read.sum + dram__bytes_write.sum of dan_stack_kernel per launch, read from the committed `ncu --set full` capture
        "traffic": traffic["per_launch"] if traffic else None, "traffic_per_candidate": traffic["per_candidate"] if traffic else None,
        "traffic_source": traffic["source"] if traffic else "no committed capture",
        "peak_source": f"{peaks['source']} bf16_tflops_sustained (kernel timed inside a long step); burst {peaks['bf16_burst']}",
        "launches_per_step": dom_launches, "avg_launch_ms": dom_ms_step / dom_launches,
        "share_of_step": dom_ms_step / sum(cls_ms.values()) if sum(cls_ms.values()) > 0 else None,
        "class_ms_per_step": cls_ms, "class_launches_per_step": cls_n,
        "whole_forward_tflops": value / world * flops_total / 1e12,
        "whole_forward_frac": (value / world * flops_total / 1e12 / peak) if peak else None,
        "hbm_frac_algorithmic": value / world * 60923 / (peaks["hbm_gbs"] * 1e9),
    }
    if args.precision == "fp32":
        # the 1e-4-parity path runs on the CUDA-core FMA pipe (DESIGN.md §4) and has no per-class event hooks: whole-forward FLOP
        # rate against the fp32 FMA peak of the part (148 SMs x 128 lanes x 2 FLOP x max SM clock)
        fma_peak, fma_src = fma_peak_tflops(clocks)
        ach = value / world * flops_total / 1e12
        roofline = {"bound": "fp32_fma (CUDA cores)", "kernel": "whole forward (sgemm_taps_kernel dominates)", "achieved": ach, "peak": fma_peak,
                    "unit": "TFLOP/s", "frac": ach / fma_peak, "traffic": None, "peak_source": fma_src}
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16" if args.precision == "bf16" else "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "candidates_per_step_per_gpu": B, "model": "PROD", "reads": R, "window": P,
                   "precision": args.precision,
                   "l2_policy": (f"inputs per step {in_bytes/1e6:.0f} MB > 126 MB L2, no flush" if in_bytes > 126e6 else
                                 f"inputs per step {in_bytes/1e6:.0f} MB; intermediates of a step ({B * 31.3:.0f} MB written and re-read) exceed the 126 MB L2, no flush"),
                   "parallelism": f"candidate-sharded x{world}, no collective"},
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": in_bytes, "d2h_bytes_per_step": B * _lib.NUM_HEAD_OUTPUTS * 4,
                "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": launches, "clocks": clocks, "roofline": roofline,
    }
    line["train"] = train_block
    if world == 1 and args.precision == "bf16" and not args.no_fp32:
        line["fp32"] = fp32_block(model, sample, dev, cfg, clocks, steps=args.steps)
    if world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        nb, reps = 64, 10                  # BASELINE.md §5: >= 640 timed candidates
        rate, times = cpu_reference_rate(cfg, sd, sample, nb, repeats=reps, warmup=1)
        line["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
                                "sample": f"{reps} timed batches x {nb} = {reps * nb} of the same dense PROD candidates (1 warm-up), torch {torch.__version__} "
                                          f"CPU fp32, oracle/dan_torch_cpu.py = the reference's op sequence; batch times {['%.2f' % t for t in times]} s"}
        if not args.no_eager_baseline:
            line["torch_eager_gpu"] = torch_eager_gpu_rate(cfg, sd, sample, dev)
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10, help="timed steps of every region that times this project's code (value, e2e, "
                    "profile pass, fp32 and train blocks); the CPU and torch-eager baseline samples keep their fixed sizes")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--batch", type=int, default=4144, help="candidates per step per GPU (28 passes of 148 candidates)")
    ap.add_argument("--pass-candidates", type=int, default=0)
    ap.add_argument("--mode", default="forward", choices=["forward", "train"], help="train: the data-parallel training step (BASELINE configs[4]) as its own line")
    ap.add_argument("--train-batch", type=int, default=32, help="candidates per training step per GPU")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-eager-baseline", action="store_true", help="skip the torch-eager-on-this-GPU sample of the reference op sequence")
    ap.add_argument("--no-fp32", action="store_true", help="skip the fp32 1e-4-parity path block (BASELINE configs[1])")
    ap.add_argument("--no-train", action="store_true", help="skip the training-step block (BASELINE configs[4])")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the head matrix of the last timed step to DIR/heads.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.mode != "forward"):
        ap.error("--dump-outputs applies to the forward benchmark of --impl b200")
    if args.impl == "reference":
        return run_reference(args)
    return run_b200(args)


if __name__ == "__main__":
    sys.exit(main())
