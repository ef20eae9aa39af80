"""ORACLE — the reference's op sequence in any dtype, on CPU or CUDA, in eval or training mode.  TEST INFRASTRUCTURE ONLY.

The same torch library calls as oracle/dan_torch_cpu.py (dl4vc/model.py:450-627 encode, :719-778 conv stack, :824-861 pool /
highway, :911-958 FC / heads), with these differences that make it a yardstick for the kernels rather than a benchmark baseline:
  * any dtype (float64 for the truth) and any device — on CUDA the caller turns TF32 off (`no_tf32`);
  * training mode: batch-statistics BatchNorm that updates the running statistics (momentum 0.1), parameters as autograd leaves;
  * the FC trunk's Dropout is the identity unless `dropout` gives p and the keep mask of every site, which the kernels draw from a
    counter-based hash (`dropout_keep` / `dropout_masks` restate it, so the same masks can be applied here);
  * `removed` replaces chosen reads by the empty-read encoding of the training kernels' read-removal augmentation, as the port documents
    it at `encode_channel` (dl4vc_b200/csrc/dan_kernels_common.cuh): token 0 in the read half, the reference half unchanged, the q,
    strand, ref-agreement, var-agreement and var_len channels zero;
  * the FC input is returned block by block (`fc_blocks`), in the reference's feature order, next to the heads.

Only tests/ import this file; dan_torch_cpu.py stays the bench baseline.
"""
from __future__ import annotations

import contextlib
from dataclasses import dataclass

import numpy as np
import torch
import torch.nn.functional as F

from dl4vc_b200.config import BN_EPS, DanConfig, HEAD_NAMES, Q_SCORE_SCALE_FACTOR, STRAND_ENCODE_FACTOR

NOT_TRAINED = ("pe", "bin_output_weights", "vt_output_weights")


@contextlib.contextmanager
def no_tf32():
    """cuDNN convolutions and cuBLAS matmuls in full fp32 / fp64 (TF32 off) for the duration of the block."""
    saved = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        yield
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = saved


class _KinkRelu(torch.autograd.Function):
    """relu whose derivative at near-zero inputs (|z| <= tol * max|z| over the tensor) is forced to `side` (1 or 0)."""

    @staticmethod
    def forward(ctx, z, tol, side):
        near = z.abs() <= tol * z.abs().amax()
        ctx.save_for_backward(((z > 0) & ~near) | (near & bool(side)))
        return z.clamp_min(0)

    @staticmethod
    def backward(ctx, g):
        (keep,) = ctx.saved_tensors
        return g * keep, None, None


class _KinkMaxReads(torch.autograd.Function):
    """max over the read axis (dim 2) whose gradient goes to the first maximum, or with side 1 to the runner-up read where that one is
    below the maximum by no more than tol * max|h| (an exact tie keeps the first read, as torch's max_pool2d and the kernels do)."""

    @staticmethod
    def forward(ctx, h, tol, side):
        first = h.argmax(dim=2, keepdim=True)
        top = h.gather(2, first)
        idx = first
        if side and h.shape[2] > 1:
            second = h.scatter(2, first, float("-inf")).argmax(dim=2, keepdim=True)
            gap = top - h.gather(2, second)
            idx = torch.where((gap > 0) & (gap <= tol * h.abs().amax()), second, first)
        ctx.save_for_backward(idx)
        ctx.shape = h.shape
        return top

    @staticmethod
    def backward(ctx, g):
        (idx,) = ctx.saved_tensors
        return torch.zeros(ctx.shape, dtype=g.dtype, device=g.device).scatter(2, idx, g), None, None


def dropout_keep(p, seed, salt, rows, ld, width):
    """(rows, width) bool: the elements dropout_kernel (dl4vc_b200/csrc/dan_train.cu) keeps at site `salt` for `seed` and probability
    `p`, over a row-major activation of leading dimension `ld` (element index b * ld + k). The hash is splitmix64's finaliser in wrapping
    uint64 arithmetic; an element is dropped when its upper 32 bits fall below min(float32(p) * 2^32, 4294967295.f) truncated to uint32."""
    i = np.arange(rows, dtype=np.uint64)[:, None] * np.uint64(ld) + np.arange(width, dtype=np.uint64)[None, :]
    x = np.uint64(seed) ^ (np.uint64(0x9E3779B97F4A7C15) * (i + np.uint64(1))) ^ (np.uint64(salt) << np.uint64(56))
    x ^= x >> np.uint64(30)
    x *= np.uint64(0xBF58476D1CE4E5B9)
    x ^= x >> np.uint64(27)
    x *= np.uint64(0x94D049BB133111EB)
    x ^= x >> np.uint64(31)
    p32 = np.float32(p)
    if not p32 > 0:
        return np.ones((rows, width), dtype=bool)
    # 4294967295.f rounds to 2^32; the device's float-to-uint32 conversion saturates there
    thr = min(int(min(p32 * np.float32(2.0 ** 32), np.float32(4294967295.0))), 0xFFFFFFFF)
    return (x >> np.uint64(32)) >= np.uint64(thr)


def dropout_masks(cfg: DanConfig, rows, p, seed):
    """The `dropout` argument of forward for one training step of the kernels: (p, keep masks of sites 0 .. len(layer_sizes)). Site 0 is
    the FC input (fc_in_features columns of rows padded to a multiple of 16, dan_capi.cu fcInPad), site j the output of FC layer j - 1."""
    widths = [cfg.fc_in_features] + list(cfg.layer_sizes)
    lds = [(cfg.fc_in_features + 15) // 16 * 16] + list(cfg.layer_sizes)
    return p, [dropout_keep(p, seed, j, rows, ld, w) for j, (ld, w) in enumerate(zip(lds, widths))]


def fc_blocks(cfg: DanConfig):
    """name -> column slice of the FC input (model.py:838-912), in order: "post_pool" (pool_combine_dimension > 0) or "max" (unless
    skip_final_maxpool) and "mean"; then "hw<l>" per conv layer (concatenated highway, 0-based l) or "hw" (averaged highway)."""
    out, k = {}, 0

    def add(name, n):
        nonlocal k
        out[name] = slice(k, k + n)
        k += n

    if cfg.pool_combine_dimension > 0:
        add("post_pool", cfg.pool_combine_dimension)
    else:
        if not cfg.skip_final_maxpool:
            add("max", cfg.channels * cfg.read_len)
        add("mean", cfg.channels * cfg.read_len)
    if cfg.highway:
        n = cfg.bottleneck * cfg.num_reads
        for l in range(cfg.total_conv_layers if cfg.concat_hw_reads else 1):
            add(f"hw{l}" if cfg.concat_hw_reads else "hw", n)
    assert k == cfg.fc_in_features
    return out


@dataclass
class RefResult:
    heads: torch.Tensor       # (B, 27) [xbinary|xVT|sigmoid(xAF)|leaky_relu(xCov)|xVB|xVR]
    fc_in: torch.Tensor       # (B, fc_in_features), reference feature order
    blocks: dict              # name -> (B, n) view of fc_in (fc_blocks)
    params: dict              # name -> tensor used (autograd leaves in training mode)
    bufs: dict                # name -> BatchNorm running buffer (updated in place in training mode)


def forward(cfg: DanConfig, sd, arrays, dtype=torch.float64, device="cpu", train=False, kink_side=None, kink_tol=3e-6,
            removed=None, dropout=None) -> RefResult:
    """The reference's forward over `arrays` = (reads, q_scores, strands, ref, ref_masks, var_masks) (PileupBatch.arrays() order) with
    the weights of state dict `sd`, computed in `dtype` on `device`.

    removed: optional (B, R) bool, reads replaced by the empty-read encoding (module docstring). dropout: optional (p, keep masks), the
    masks of the nn.Dropout sites of conv2hidden in order (the FC input, then the output of every FC ReLU), each (B, width) bool
    (dropout_masks); kept values are scaled by 1 / (1 - p).

    kink_side 0 / 1: same values, but every ReLU whose input is within kink_tol of zero (relative to its tensor's largest |input|), and
    the read-axis max where the runner-up read is within kink_tol of the maximum, backpropagates as if it sat on the off / on side of the
    kink. An fp32 computation of the same values can land on either side there, so the two gradients bound how far an fp32 gradient may
    legitimately be from the float64 one (kink_bound). The default kink_tol, 3e-6, is the fp32 kernels' measured forward accuracy (worst
    FC-input block 2.9e-6 of its largest value, tests/test_gpu_config_space.py)."""
    dev = torch.device(device)
    relu = F.relu if kink_side is None else (lambda z: _KinkRelu.apply(z, kink_tol, kink_side))
    params = {k: torch.as_tensor(v).to(dev, dtype).clone().requires_grad_(train) for k, v in sd.items()
              if k not in NOT_TRAINED and "running_" not in k and "num_batches" not in k}
    bufs = {k: torch.as_tensor(v).to(dev, dtype).clone() for k, v in sd.items() if "running_" in k}
    reads, q_scores, strands, ref, ref_masks, var_masks = (torch.from_numpy(np.ascontiguousarray(a)).to(dev) for a in arrays)
    reads, ref = reads.long(), ref.long()
    gone = None if removed is None else torch.as_tensor(np.asarray(removed, dtype=bool)).to(dev)
    if gone is not None:
        reads = reads.masked_fill(gone.unsqueeze(1), 0)                                    # token 0: counted as padding
    E, pe = params["embeddings.weight"], torch.as_tensor(sd["pe"]).to(dev, dtype)
    B, P, R = reads.shape
    # ---- encode (model.py:450-627); nn.Embedding(padding_idx=0, scale_grad_by_freq=True) of model.py:143-145 ----
    reads_emb = F.embedding(reads, E, padding_idx=0, scale_grad_by_freq=True) + pe.unsqueeze(2)
    ref_emb = (F.embedding(ref, E, padding_idx=0, scale_grad_by_freq=True) + pe).unsqueeze(2).expand(-1, -1, R, -1)
    x = torch.cat((reads_emb, ref_emb), dim=3)
    if cfg.use_q_scores:
        x = torch.cat((x, (q_scores.to(dtype) * Q_SCORE_SCALE_FACTOR).unsqueeze(3)), dim=3)
    if cfg.use_strands:
        x = torch.cat((x, (strands.to(dtype) * STRAND_ENCODE_FACTOR).unsqueeze(3)), dim=3)
    if cfg.use_reads_ref_var_mask:
        chans, nzs = [], []
        for m in (ref_masks, var_masks):
            m = m.long().unsqueeze(2)
            nz = (m != 0).long()
            agree = ((reads * nz) == m).long().sum(dim=1) == P                                # model.py:592-593
            chans.append((nz * agree.unsqueeze(1).long()).to(dtype))
            nzs.append(nz)
        chans.append(nzs[0].expand(-1, -1, R).to(dtype))                                       # var_len from the REF mask (sic)
        x = torch.cat([x] + [c.unsqueeze(3) for c in chans], dim=3)
    if gone is not None:                       # every channel behind the two embedding halves is zero on a removed read, var_len too
        D = E.shape[1]
        x = torch.cat((x[..., :2 * D], x[..., 2 * D:] * (~gone).to(dtype)[:, None, :, None]), dim=3)
    h = x.permute(0, 3, 2, 1)                                                                  # (B, Cin, R, P), model.py:719
    # ---- conv stack (model.py:728-778) ----
    pool, hw, res_i = None, [], 0
    for l in range(1, cfg.total_conv_layers + 1):
        resid = h
        if pool is not None:
            h = h + pool
            pool = None
        d = cfg.dilation(l)
        h = relu(F.conv2d(h, params[f"conv1D_layers.{l-1}.weight"], params[f"conv1D_layers.{l-1}.bias"], padding=(0, d), dilation=d))
        if cfg.use_batchnorm:
            p = f"bn1D_layers.{l-1}."
            h = F.batch_norm(h, bufs[p + "running_mean"], bufs[p + "running_var"], params[p + "weight"], params[p + "bias"],
                             training=train, momentum=0.1, eps=BN_EPS)
        if cfg.is_residual(l):
            h = F.conv2d(h, params[f"residual_conv_layers.{res_i}.weight"], params[f"residual_conv_layers.{res_i}.bias"]) + resid
            res_i += 1
        if l in cfg.conv_1d_pool_layers:
            pool = F.avg_pool2d(h, kernel_size=(R, 1), ceil_mode=True)
        if cfg.highway:
            t = relu(F.conv2d(h, params[f"conv1D_bottleneck_layers.{l-1}.weight"], params[f"conv1D_bottleneck_layers.{l-1}.bias"]))
            o = F.conv2d(t, params[f"conv1D_compression_layers.{l-1}.weight"], params[f"conv1D_compression_layers.{l-1}.bias"])
            hw.append(o.reshape(B, -1))
    # ---- read-axis pooling (model.py:824-844) ----
    mean = F.avg_pool2d(h, kernel_size=(R, 1), ceil_mode=True)
    if cfg.skip_final_maxpool:
        pooled = mean.reshape(B, -1)
    else:
        mx = F.max_pool2d(h, kernel_size=(R, 1), ceil_mode=True) if kink_side is None else _KinkMaxReads.apply(h, kink_tol, kink_side)
        pooled = torch.cat((mx, mean), dim=1).reshape(B, -1)
    if cfg.pool_combine_dimension > 0:
        pooled = relu(F.linear(pooled, params["post_pool_conv1D.weight"], params["post_pool_conv1D.bias"]))
    if cfg.highway:
        hwv = torch.cat(hw, dim=1) if cfg.concat_hw_reads else torch.stack(hw, 0).mean(0)
        pooled = torch.cat((pooled, relu(hwv)), dim=1)
    fc_in = pooled
    # ---- FC trunk + heads (model.py:911-958); Dropout is the identity unless its masks are given ----
    if dropout is not None:
        p, keeps = dropout
        assert len(keeps) == len(cfg.fc_indices) + 1, "one keep mask per Dropout site"
        drop = lambda z, j: z * (torch.as_tensor(np.asarray(keeps[j], dtype=bool)).to(dev, dtype) / (1.0 - p))
    else:
        drop = lambda z, j: z
    xh = drop(fc_in, 0)
    for j, idx in enumerate(cfg.fc_indices):
        xh = drop(relu(F.linear(xh, params[f"conv2hidden.{idx}.weight"], params[f"conv2hidden.{idx}.bias"])), j + 1)
    outs = [F.linear(xh, params[n + ".weight"], params[n + ".bias"]) for n in HEAD_NAMES]
    outs[2] = torch.sigmoid(outs[2])
    outs[3] = F.leaky_relu(outs[3], 0.01)
    blocks = {name: fc_in[:, sl] for name, sl in fc_blocks(cfg).items()}
    return RefResult(torch.cat(outs, dim=1), fc_in, blocks, params, bufs)


def train_reference(cfg: DanConfig, sd, arrays, dtype, dev, kink_side=None, removed=None, dropout=None):
    """Training-mode forward (batch-statistics BatchNorm with running-statistics update; dropout and read removal as forward takes them)
    under torch autograd. Returns heads, {name: leaf parameter} and {name: updated running buffer}."""
    r = forward(cfg, sd, arrays, dtype=dtype, device=dev, train=True, kink_side=kink_side, removed=removed, dropout=dropout)
    return r.heads, r.params, r.bufs


def kink_bound(cfg: DanConfig, sd, arrays, dheads, dev, removed=None, dropout=None):
    """name -> |grad(kink_side=1) - grad(kink_side=0)| in float64: how much the gradient of each parameter moves when the ReLUs and
    read-axis maxima that sit within rounding distance of their kink switch sides. A single such unit that an fp32 forward puts on the
    other side than float64 does moves a gradient tensor by exactly this much, which no arithmetic accuracy bounds."""
    g = []
    for side in (0, 1):
        heads, params, _ = train_reference(cfg, sd, arrays, torch.float64, dev, kink_side=side, removed=removed, dropout=dropout)
        (heads * dheads.to(heads.device, torch.float64)).sum().backward()
        g.append({k: v.grad for k, v in params.items() if v.grad is not None})
    return {k: (g[1][k] - g[0][k]).abs().cpu().numpy() for k in g[0]}
