"""Speed of the MIN configuration (argparse defaults, SURVEY App. D: pool_combine_dimension 2048, FC 1024/256, no highway) on the GPU.

One run measures, with CUDA events after warm-up:
  * inference at bf16 (tcgen05 path) and at fp32 (CUDA-core path), resident uint8 inputs, --batch candidates per call;
  * one training step at --train-batch candidates: training-mode forward, device loss block, native backward, clip_grad_norm 1.0, Adam;
and prints one JSON line with candidates/s, ms per step, the device name and its power limit (--out also writes it to a file).

    python scripts/bench_pool_combine.py --batch 2072 --steps 5 --warmup 2
"""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def power_limit_w(index: int = 0):
    try:
        import pynvml
        pynvml.nvmlInit()
        return pynvml.nvmlDeviceGetPowerManagementLimit(pynvml.nvmlDeviceGetHandleByIndex(index)) / 1000.0
    except Exception:
        return None


def timed_ms(fn, steps):
    import torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--batch", type=int, default=2072, help="candidates per inference call (2072 = two FC chunks of 7 x 148)")
    ap.add_argument("--steps", type=int, default=5, help="timed inference calls per precision")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--train-batch", type=int, default=32)
    ap.add_argument("--train-steps", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if args.steps < 1 or args.train_steps < 1 or args.warmup < 0:
        ap.error("--steps and --train-steps must be >= 1, --warmup >= 0")

    import numpy as np
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_pool_combine.py measures on a CUDA device; none is visible")
    from dl4vc_b200.config import min_config
    from dl4vc_b200.factory import build_model
    from dl4vc_b200.losses import fused_losses
    from dl4vc_b200.synth import make_pileups
    from dl4vc_b200.weights import synth_state_dict

    dev = torch.device("cuda", 0)
    cfg = min_config()
    sd = synth_state_dict(cfg, seed=1)
    batch = make_pileups(args.batch, seed=2026, coverage="poisson")
    r, q, s, ref, rm, vm = (torch.from_numpy(np.ascontiguousarray(a)).to(dev) for a in batch.arrays())
    model = build_model(cfg, sd, device=dev)

    result = {"config": "MIN (min_config(): pool_combine_dimension 2048, layer_sizes 1024/256, 5 conv layers, no highway, no BatchNorm)",
              "device": torch.cuda.get_device_name(dev), "power_limit_w": power_limit_w(dev.index), "batch": args.batch, "steps": args.steps,
              "warmup": args.warmup, "inputs": "resident uint8 device tensors"}
    heads = {}
    for prec in ("bf16", "fp32"):
        model.set_precision(prec)

        def call():
            heads[prec] = model.forward_heads(r, ref, q, s, rm, vm)

        for _ in range(args.warmup):
            call()
        ms = timed_ms(call, args.steps)
        result[prec] = {"candidates_per_s": round(args.batch * args.steps / (ms * 1e-3), 1), "ms_per_call": round(ms / args.steps, 3),
                        "launches_per_call": model.last_launch_count}
    a, b = heads["bf16"].double(), heads["fp32"].double()
    result["bf16_vs_fp32_max_err_of_max_abs_logit"] = float((a - b).abs().max() / b.abs().max())
    del model, heads
    torch.cuda.empty_cache()

    # ---- one training step (fp32 kernels) ----
    model = build_model(cfg, sd, device=dev, precision="fp32").train()
    opt = torch.optim.Adam(model.parameters(), lr=2e-4)
    tb_ = make_pileups(args.train_batch, seed=4242, coverage="poisson")
    d = [torch.from_numpy(np.ascontiguousarray(x)).to(dev) for x in tb_.arrays()]
    vt = torch.from_numpy(np.rint(tb_.var_fraction * 2).astype(np.int64)).to(dev)
    tb = (vt > 0).long()
    af = torch.from_numpy(tb_.var_fraction.astype(np.float32)).to(dev)
    cov = torch.from_numpy((tb_.num_reads * 0.01).astype(np.float32)).to(dev)
    vb = torch.from_numpy(tb_.var_masks[:, 100].astype(np.int64)).to(dev)
    vr = torch.from_numpy(tb_.ref_masks[:, 100].astype(np.int64)).to(dev)

    def step():
        opt.zero_grad(set_to_none=True)
        h = model.forward_train_heads(d[0], d[3], d[1], d[2], d[4], d[5])
        total, _, _, _ = fused_losses(h, tb, vt, af, cov, vb, vr)
        total.backward()
        torch.nn.utils.clip_grad_norm_(model.parameters(), 1.0)
        opt.step()

    for _ in range(max(args.warmup, 1)):
        step()
    ms = timed_ms(step, args.train_steps)
    result["train"] = {"batch": args.train_batch, "steps": args.train_steps, "ms_per_step": round(ms / args.train_steps, 3),
                       "candidates_per_s": round(args.train_batch * args.train_steps / (ms * 1e-3), 1),
                       "step": "train forward + dan_losses + dan_backward + clip_grad_norm 1.0 + Adam (one GPU, dropout 0 as in MIN)"}
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
