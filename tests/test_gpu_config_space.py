"""The kernels across the configuration space DESIGN.md §1 says they take, against the reference's op sequence in float64.

Every case of CASES is a small_config / min_config override; its comment names the kernel branch it reaches. For each case the fp32
path, the bf16 path (on the route the table expects: fused conv-stack kernel, layer by layer, or a rejection naming the reason) and,
where the fused kernel runs, the layer-by-layer route on the same inputs are compared with oracle/dan_torch_ref.py in float64 on the
GPU (TF32 off): the heads, and the FC input block by block (pooled max, mean, each layer's highway slice, the post-pool output), each
block against its own largest value. Candidates mix Poisson, full and empty coverage. A second table runs one training step per case
against float64 autograd.

Bars (the max over candidates of |kernel - float64|, divided by the block's largest |float64| value):
  fp32 heads 1e-4 of the largest |logit| (tests/test_gpu_parity.py), fp32 FC-input blocks 1e-4;
  bf16 heads 3e-2, bf16 FC-input blocks 2e-2, fused vs layer-by-layer blocks 2e-2.
Measured on B200 (DESIGN.md §2 lists the figures): fp32 blocks <= 3e-6; bf16 blocks up to 1.9e-2 on the goldens and on the sweep, so
the 2e-2 bar has little headroom — it is the bar of the existing FC-input tests, applied per block instead of per vector.
"""
import dataclasses
import json

import numpy as np
import pytest
import torch

from conftest import GOLDEN_CASES, load_golden, rel_err
from dl4vc_b200.config import min_config, small_config
from dl4vc_b200.factory import build_model
from dl4vc_b200.synth import make_pileups
from dl4vc_b200.weights import synth_state_dict
from oracle import dan_torch_ref

FP32_TOL = 1e-4          # heads and FC-input blocks
BF16_TOL = 3e-2          # heads
BF16_BLOCK_TOL = 2e-2    # FC-input blocks, bf16 vs float64 and fused vs layer by layer
GRAD_TOL = 5e-3          # training: per tensor, relative to its largest |gradient| (tests/test_gpu_pool_combine.py)
F, L = "fused", "layerwise"
ROUTE_CODE = {F: 1, L: 2}

# id, configuration, bf16 route: F (fused dan_stack_kernel), L (dan_layer_kernel per layer) or the reason the bf16 path rejects it
CASES = [
    # ---- read counts: PROD topology, the fused kernel encodes layer 1 itself; work goes out in blocks of 20 reads (dan_stack.cuh StkIter)
    ("reads1", small_config(num_reads=1), F),                 # one block of one read: phantom slot-1 read, no slot-1 sum group
    ("reads2", small_config(num_reads=2), F),                 # one block of one read pair
    ("reads3", small_config(num_reads=3), F),                 # odd block: phantom read in the second pair
    ("reads19", small_config(num_reads=19), F),               # one odd block short of 20
    ("reads21", small_config(num_reads=21), F),               # full block + a one-read block (group_mean8 skips its slot-1 group)
    ("reads41", small_config(num_reads=41), F),               # two full blocks + a one-read block
    ("reads99", small_config(num_reads=99), F),               # four full blocks + an odd 19-read block
    # ---- input channel sets: the separate bf16 encoder (encode_rows_bf16_kernel) feeds layer 1 as kc_in planes (kStkInPlanes)
    ("in16", small_config(embed_dim=4, use_q_scores=False, use_strands=False, use_reads_ref_var_mask=False), F),   # Cin 8 -> 16
    ("in32", small_config(embed_dim=8), F),                   # Cin 21 -> 32
    ("in48_no_q", small_config(use_q_scores=False), F),       # Cin 44 -> 48, not the shipped set
    ("in48_no_masks", small_config(use_reads_ref_var_mask=False), F),   # Cin 42 -> 48
    ("in80", small_config(embed_dim=32), F),                  # Cin 69 -> 80
    ("in128", small_config(embed_dim=60), F),                 # Cin 125 -> 128, the widest layer-1 tile (an odd embed_dim has no
                                                              # sinusoidal table: model.py's pe construction needs an even width)
    ("in144", small_config(embed_dim=64), "more than 128 padded input channels"),   # Cin 133 -> 144
    # ---- dilation: the fused kernel's read buffer has kStkLead = 2 zero rows, the layer-wise tiles a halo of up to 8
    ("dil1_2", small_config(middle_layer_dilation=1, final_layer_dilation=2), F),
    ("dil2_1", small_config(middle_layer_dilation=2, final_layer_dilation=1), F),
    ("dil3_3", small_config(middle_layer_dilation=3, final_layer_dilation=3), L),
    ("dil2_8", small_config(middle_layer_dilation=2, final_layer_dilation=8), L),
    # ---- layer count and segments (kStkMaxSeg = 8 layers per fused launch; a pool-add ends a segment)
    ("L1", small_config(total_conv_layers=1, conv_1d_pool_layers=(), residual_layer_start=0), F),
    ("L2_pool1", small_config(total_conv_layers=2, conv_1d_pool_layers=(1,), residual_layer_start=0), F),   # two one-layer segments
    ("L10_seg8", small_config(total_conv_layers=10), F),      # pool (2,), residual from 5: segment 3-10 has 8 layers
    ("L11_seg9", small_config(total_conv_layers=11), L),      # segment 3-11 has 9
    ("L12_nopool", small_config(total_conv_layers=12, conv_1d_pool_layers=()), L),
    ("L12_pools4_8", small_config(total_conv_layers=12, conv_1d_pool_layers=(4, 8), residual_layer_start=0), F),   # three segments
    # ---- pool-add / residual placement
    ("pools2_4_res6", small_config(conv_1d_pool_layers=(2, 4), residual_layer_start=6), F),   # two bias maps
    ("pool_last", small_config(conv_1d_pool_layers=(7,)), F),  # pool after the last layer: computed, never consumed
    ("res2_nopool", small_config(residual_layer_start=2, conv_1d_pool_layers=()), F),
    ("res2_pool2", small_config(residual_layer_start=2), L),  # layer 3: residual directly behind the pool-add
    # ---- highway and head
    ("bn_off_highway", small_config(use_batchnorm=False), F),
    ("hw_averaged", small_config(concat_hw_reads=False), F),
    ("skip_max_highway", small_config(skip_final_maxpool=True), F),
    ("bott64", small_config(bottleneck=64), L),
    ("bott16", small_config(bottleneck=16), "bottleneck must be 32 or 64"),
    ("bott48", small_config(bottleneck=48), "bottleneck must be 32 or 64"),
    ("d64_reads21", small_config(pool_combine_dimension=64, num_reads=21), F),   # post-pool GEMM behind a one-read block
    # ---- widths: the bf16 kernels are built for 128 channels and FC widths that are multiples of 32
    ("C16", small_config(channels=16), "128 conv channels"),
    ("C32", small_config(channels=32), "128 conv channels"),
    ("C64", small_config(channels=64), "128 conv channels"),
    ("fc48", small_config(layer_sizes=(48,)), "FC widths must be multiples of 32"),
    ("fc32", small_config(layer_sizes=(32,)), F),
    ("fc64_32_32_32", small_config(layer_sizes=(64, 32, 32, 32)), F),
    ("min_fc32", min_config(layer_sizes=(32,), pool_combine_dimension=64), F),   # MIN topology, separate encoder (40 channels)
]


def _tensors(arrays):
    return [torch.from_numpy(np.ascontiguousarray(a)) for a in arrays]


def _heads(model, arrays):
    r, q, s, ref, rm, vm = _tensors(arrays)
    return model.forward_heads(r, ref, q, s, rm, vm).cpu().numpy()


def _batch(R, seed):
    """6 candidates: 3 Poisson depth (clipped to [1, R]), 2 full, 1 without reads."""
    parts = [make_pileups(3, seed=seed, num_reads=R, coverage="poisson"), make_pileups(2, seed=seed + 1, num_reads=R, coverage="full"),
             make_pileups(1, seed=seed + 2, num_reads=R, coverage="empty")]
    return tuple(np.concatenate(a, axis=0) for a in zip(*(p.arrays() for p in parts)))


def _reference(cfg, sd, arrays):
    with dan_torch_ref.no_tf32():
        r = dan_torch_ref.forward(cfg, sd, arrays, dtype=torch.float64, device="cuda")
    return r.heads.cpu().numpy(), r.fc_in.cpu().numpy()


def _block_errs(cfg, got, want):
    """name -> max |got - want| over the block / max |want| of the block (FC input in the reference's feature order)."""
    assert got.shape == want.shape, (got.shape, want.shape)
    out = {}
    for name, sl in dan_torch_ref.fc_blocks(cfg).items():
        w = want[:, sl]
        out[name] = float(np.abs(got[:, sl] - w).max() / max(np.abs(w).max(), 1e-30))
    return out


def _fc_input(model, arrays):
    heads = _heads(model, arrays)
    return heads, model.debug_fc_input(len(arrays[0])).cpu().numpy()


def _check_blocks(fails, errs, tag, block_errs, tol):
    for name, e in block_errs.items():
        errs[f"{tag}/{name}"] = e
        if not e < tol:
            fails.append(f"{tag} block {name}: {e:.3e} >= {tol:g}")


def _split_bitwise(model, arrays, full, tag, fails):
    """Candidates are independent: a batch cut in two (not at an internal pass boundary) gives bitwise the same rows."""
    n = len(arrays[0])
    parts = np.concatenate([_heads(model, tuple(a[lo:hi] for a in arrays)) for lo, hi in ((0, 2 * n // 3), (2 * n // 3, n))])
    if not np.array_equal(parts, full):
        fails.append(f"{tag}: batch split changes the heads (max diff {np.abs(parts - full).max():.3e})")


def _run_case(cfg, route, seed, arrays=None):
    sd = synth_state_dict(cfg, seed=seed)
    arrays = _batch(cfg.num_reads, seed + 10) if arrays is None else arrays
    want_heads, want_fc = _reference(cfg, sd, arrays)
    fails, errs = [], {}

    model = build_model(cfg, sd, precision="fp32")
    h32, fc32 = _fc_input(model, arrays)
    errs["fp32/heads"] = rel_err(h32, want_heads)
    if not errs["fp32/heads"] < FP32_TOL:
        fails.append(f"fp32 heads: {errs['fp32/heads']:.3e}")
    _check_blocks(fails, errs, "fp32", _block_errs(cfg, fc32, want_fc), FP32_TOL)
    _split_bitwise(model, arrays, h32, "fp32", fails)

    got_route = model.bf16_route()
    model.set_precision("bf16")
    if route not in ROUTE_CODE:
        assert got_route == 0, f"bf16 route {got_route}, expected a rejection ({route})"
        with pytest.raises(NotImplementedError, match=route):
            _heads(model, arrays)
        assert np.array_equal(_heads(model.set_precision("fp32"), arrays), h32), "fp32 after the bf16 rejection"
        return fails, errs
    assert got_route == ROUTE_CODE[route], f"bf16 route {got_route}, expected {ROUTE_CODE[route]} ({route})"
    h16, fc16 = _fc_input(model, arrays)
    assert np.isfinite(h16).all() and np.isfinite(fc16).all()
    errs["bf16/heads"] = rel_err(h16, want_heads)
    if not errs["bf16/heads"] < BF16_TOL:
        fails.append(f"bf16 heads: {errs['bf16/heads']:.3e}")
    _check_blocks(fails, errs, "bf16", _block_errs(cfg, fc16, want_fc), BF16_BLOCK_TOL)
    _split_bitwise(model, arrays, h16, "bf16", fails)
    if route == F:
        model.set_layerwise(True)
        assert model.bf16_route() == ROUTE_CODE[L]
        hl, fcl = _fc_input(model, arrays)
        errs["layerwise/heads"] = rel_err(hl, want_heads)
        if not errs["layerwise/heads"] < BF16_TOL:
            fails.append(f"layer-wise heads: {errs['layerwise/heads']:.3e}")
        _check_blocks(fails, errs, "fused_vs_layerwise", _block_errs(cfg, fc16, fcl), BF16_BLOCK_TOL)
    return fails, errs


def _report(name, errs):
    print(f"\nSWEEP {name} " + json.dumps({k: float(f"{v:.3e}") for k, v in errs.items()}))


# ---------------------------------------------------------------------------------------------------------------- inference
@pytest.mark.gpu
@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_per_block_bars_hold_on_reference_goldens(name):
    """The per-block bars on the six configurations the real reference was run on (tests/golden), as the sweep applies them."""
    g = load_golden(name)
    cfg = g["cfg"]
    route = L if cfg.conv_1d_pool_layers == (1, 3) else F        # variant_a: residual layer 4 behind the pool-add after layer 3
    fails, errs = _run_case(cfg, route, g["seed"], g["arrays"])
    _report("golden:" + name, errs)
    assert not fails, fails


@pytest.mark.gpu
@pytest.mark.parametrize("name,cfg,route", CASES, ids=[c[0] for c in CASES])
def test_config_space_matches_float64_reference(name, cfg, route):
    fails, errs = _run_case(cfg, route, seed=sum(map(ord, name)))
    _report(name, errs)
    assert not fails, fails


@pytest.mark.gpu
def test_dilation_above_8_is_rejected_when_the_model_is_created():
    cfg = small_config(middle_layer_dilation=9)
    model = build_model(cfg, synth_state_dict(cfg, seed=1), precision="fp32")
    with pytest.raises(NotImplementedError, match="dilation 9"):
        _heads(model, make_pileups(1, seed=1).arrays())


@pytest.mark.gpu
@pytest.mark.parametrize("route", ["fp32", F, L])
def test_read_blocks_count_every_read_once(route):
    """Without pool-adds and highway each read's activations depend on that read alone and no weight depends on num_reads. 21 reads
    leave a one-read block with a phantom read; duplicating them (42 reads: two full blocks and a two-read one) must leave the read-axis
    max bitwise unchanged and the mean and heads within the bars."""
    base = small_config(conv_1d_pool_layers=(), highway=False)
    c21, c42 = small_config(conv_1d_pool_layers=(), highway=False, num_reads=21), small_config(conv_1d_pool_layers=(), highway=False, num_reads=42)
    sd = synth_state_dict(base, seed=31)
    a21 = _batch(21, 32)
    a42 = tuple(np.concatenate([a, a], axis=2) if a.ndim == 3 else a for a in a21)
    out = {}
    for cfg, arrays in ((c21, a21), (c42, a42)):
        model = build_model(cfg, sd, precision="fp32" if route == "fp32" else "bf16")
        if route != "fp32":
            model.set_layerwise(route == L)
            assert model.bf16_route() == ROUTE_CODE[route]
        out[cfg.num_reads] = _fc_input(model, arrays)
    blocks = dan_torch_ref.fc_blocks(c21)
    (h21, f21), (h42, f42) = out[21], out[42]
    assert np.array_equal(f21[:, blocks["max"]], f42[:, blocks["max"]]), "read-axis max"
    tol_block, tol_heads = (FP32_TOL, FP32_TOL) if route == "fp32" else (BF16_BLOCK_TOL, BF16_TOL)
    mean = f42[:, blocks["mean"]]
    err = np.abs(f21[:, blocks["mean"]] - mean).max() / np.abs(mean).max()
    print(f"\nREADBLOCKS {route} mean {err:.3e} heads {rel_err(h21, h42):.3e}")
    assert err < tol_block, f"read-axis mean off by {err:.3e}"
    assert rel_err(h21, h42) < tol_heads


# ---------------------------------------------------------------------------------------------------------------- training
TRAIN_CASES = [
    ("reads1", small_config(num_reads=1)),
    ("reads21", small_config(num_reads=21)),
    ("in32", small_config(embed_dim=8)),
    ("in144", small_config(embed_dim=64)),                     # CinPad 144 > C: d(x0) is wider than a conv row
    ("C32", small_config(channels=32)),                        # CinPad 48 > C = 32
    ("dil3_8", small_config(middle_layer_dilation=3, final_layer_dilation=8)),
    ("L1", small_config(total_conv_layers=1, conv_1d_pool_layers=(), residual_layer_start=0)),
    ("L12_pools4_8", small_config(total_conv_layers=12, conv_1d_pool_layers=(4, 8), residual_layer_start=0)),
    ("pools1_3", small_config(conv_1d_pool_layers=(1, 3), residual_layer_start=0)),
    ("bn_off_highway", small_config(use_batchnorm=False)),
    ("hw_averaged_skip_max", small_config(concat_hw_reads=False, skip_final_maxpool=True)),
    ("bott16", small_config(bottleneck=16)),
    ("bott64", small_config(bottleneck=64)),
    ("fc32", small_config(layer_sizes=(32,))),
    ("fc64_32_32_32", small_config(layer_sizes=(64, 32, 32, 32))),
]


def _sampled(a, above=200_000, stride=97):
    a = np.asarray(a, np.float64)
    return a.reshape(-1)[::stride] if a.size > above else a


def _train_reference(cfg, sd, arrays, cw, removed=None, dropout=None):
    """One training step of oracle/dan_torch_ref.py on the GPU (TF32 off) with d(loss)/d(heads) = cw: {dtype: (heads, gradients, running
    buffers)} for float64 and float32, and the kink bound of every gradient. removed / dropout: as dan_torch_ref.forward takes them."""
    ref = {}
    with dan_torch_ref.no_tf32():
        for dtype in (torch.float64, torch.float32):
            heads, params, bufs = dan_torch_ref.train_reference(cfg, sd, arrays, dtype, "cuda", removed=removed, dropout=dropout)
            (heads * torch.from_numpy(cw).to(heads.device, dtype)).sum().backward()
            grads = {k: v.grad.cpu().numpy() for k, v in params.items() if v.grad is not None}
            ref[dtype] = (heads.detach().cpu().numpy(), grads, {k: v.cpu().numpy() for k, v in bufs.items()})
        kink = dan_torch_ref.kink_bound(cfg, sd, arrays, torch.from_numpy(cw), "cuda", removed=removed, dropout=dropout)
    return ref, kink


def _train_step(model, arrays, cw, **kw):
    """One training step of the kernels through model(...) with d(loss)/d(heads) = cw; kw: rm_non_var_reads / rm_var_reads."""
    r, q, s, rf, rm, vm = (t.long() for t in _tensors(arrays))
    dummy = torch.zeros(len(arrays[0]), dtype=torch.long)
    out = model(r, rf, q, s, dummy, dummy, dummy, dummy, rm, vm, **kw)
    heads = torch.cat([o.reshape(o.shape[0], -1) for o in out[:6]], dim=1)
    (heads * torch.from_numpy(cw).to(heads.device)).sum().backward()
    return heads.detach().cpu().numpy()


def _check_train_step(name, model, heads, ref, kink):
    """The heads, every gradient tensor and the running statistics of `model` after _train_step against _train_reference."""
    want_heads, want_grads, want_bufs = ref[torch.float64]
    assert rel_err(heads, want_heads) < FP32_TOL, "training-mode forward"

    # The gradient is discontinuous where a ReLU input or the read-axis max sits at its kink: a unit within rounding distance of it can
    # land on either side in fp32 and move a gradient tensor by 1e-2 of its maximum (measured: with 21 reads the kernels' layer-4 bottleneck
    # weight gradient is 1.4e-2 off float64, exactly what the ReLUs of that layer within 1e-6 of their kink account for). kink_bound says, element by element, how far such
    # units can move each gradient; beyond that, the bar of tests/test_gpu_pool_combine.py holds: 5e-3 of the tensor's largest |gradient|,
    # or 1.5x what torch's own fp32 autograd achieves on an ill-conditioned tensor.
    errs, beyond, own, bad = {}, {}, {}, {}
    for pname, p in model.named_parameters():
        if pname not in want_grads:
            assert p.grad is None or pname in dan_torch_ref.NOT_TRAINED, pname
            continue
        assert p.grad is not None, f"no gradient for {pname}"
        got, want, kb = _sampled(p.grad.detach().cpu().numpy()), _sampled(want_grads[pname]), _sampled(kink[pname])
        scale = max(np.abs(want).max(), 1e-20)
        errs[pname] = float(np.abs(got - want).max() / scale)
        own[pname] = float(np.abs(_sampled(ref[torch.float32][1][pname]) - want).max() / scale)
        beyond[pname] = float((np.abs(got - want) - kb).max() / scale)
        if not beyond[pname] < max(GRAD_TOL, 1.5 * own[pname]):
            bad[pname] = (errs[pname], beyond[pname], own[pname])
    assert len(errs) == len(want_grads)
    worst = max(errs, key=errs.get)
    print(f"\nTRAIN {name} worst {worst} {errs[worst]:.2e} (beyond the kink bound {beyond[worst]:.2e}, fp32 autograd {own[worst]:.2e}); "
          f"worst beyond the kink bound {max(beyond.values()):.2e}")
    assert not bad, f"gradients off (error, error beyond the kink bound, fp32 autograd error): {bad}"
    for bname, b in model.named_buffers():
        if "running_" in bname:
            np.testing.assert_allclose(b.detach().cpu().numpy(), want_bufs[bname], rtol=2e-5, atol=1e-6, err_msg=bname)


@pytest.mark.gpu
@pytest.mark.parametrize("name,cfg", TRAIN_CASES, ids=[c[0] for c in TRAIN_CASES])
def test_training_step_matches_float64_autograd(name, cfg):
    cfg = dataclasses.replace(cfg, hidden_dropout=0.0)          # dropout: tests/test_gpu_train_dropout_removal.py
    seed = sum(map(ord, name))
    sd = synth_state_dict(cfg, seed=seed)
    arrays = tuple(a[[0, 1, 3, 5]] for a in _batch(cfg.num_reads, seed + 1))       # 2 Poisson, 1 full, 1 empty
    cw = np.random.default_rng(seed + 2).standard_normal((len(arrays[0]), 27)).astype(np.float32)
    ref, kink = _train_reference(cfg, sd, arrays, cw)
    model = build_model(cfg, sd, precision="fp32").train()
    _check_train_step(name, model, _train_step(model, arrays, cw), ref, kink)


@pytest.mark.gpu
def test_training_rejects_a_residual_layer_behind_a_pool_add_before_touching_state():
    """variant_a's topology (pool after layer 3, residual layer 4): the gradient of such a layer is not implemented, so the training
    forward raises before it updates the BatchNorm running statistics."""
    cfg = load_golden("variant_a")["cfg"]
    model = build_model(cfg, synth_state_dict(cfg, seed=3), precision="fp32").train()
    before = {k: v.detach().clone() for k, v in model.named_buffers() if "running_" in k or "num_batches" in k}
    r, q, s, rf, rm, vm = (t.long() for t in _tensors(make_pileups(2, seed=4, coverage="poisson").arrays()))
    dummy = torch.zeros(2, dtype=torch.long)
    with pytest.raises(NotImplementedError, match="residual layer directly behind a pool-add"):
        model(r, rf, q, s, dummy, dummy, dummy, dummy, rm, vm)
    after = dict(model.named_buffers())
    for k, v in before.items():
        assert torch.equal(after[k], v), k
