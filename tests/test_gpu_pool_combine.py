"""pool_combine_dimension (post_pool_conv1D, model.py:841-843) on the bf16 tensor-core path and in training.

GPU tests (-m gpu) run the kernels against the real reference's goldens, the fp32 path, the numpy oracle and torch autograd over the
op sequence of oracle/dan_torch_ref.py in float64; the bucket test runs on the CPU."""
import numpy as np
import pytest
import torch

from conftest import load_golden, rel_err
from dl4vc_b200.config import min_config, small_config
from dl4vc_b200.factory import build_model, ctor_kwargs
from dl4vc_b200.synth import make_pileups
from dl4vc_b200.weights import synth_state_dict
from oracle import dan_oracle, dan_torch_ref

BF16_TOL = 3e-2          # the bf16 bar of tests/test_gpu_parity.py: heads within 3e-2 of the largest |logit|
GRAD_TOL = 5e-3          # the training bar of tests/test_gpu_train.py: per tensor, relative to its largest |gradient|
SAMPLE_ABOVE, SAMPLE_STRIDE = 200_000, 97


def _tensors(arrays):
    return [torch.from_numpy(np.ascontiguousarray(a)) for a in arrays]


def _heads(model, arrays):
    r, q, s, ref, rm, vm = _tensors(arrays)
    return model.forward_heads(r, ref, q, s, rm, vm).cpu().numpy()


def _bf16_vs_fp32(cfg, n, seed):
    sd = synth_state_dict(cfg, seed=seed)
    batch = make_pileups(n, seed=seed + 100, coverage="poisson")
    model = build_model(cfg, sd, precision="fp32")
    ref32 = _heads(model, batch.arrays())
    got = _heads(model.set_precision("bf16"), batch.arrays())
    assert np.isfinite(got).all()
    return rel_err(got, ref32)


# ---------------------------------------------------------------------------------------------------------------- bf16 inference
@pytest.mark.gpu
def test_bf16_min_smallfc_matches_reference_golden():
    g = load_golden("min_smallfc")
    cfg = g["cfg"]
    assert cfg.pool_combine_dimension > 0
    model = build_model(cfg, synth_state_dict(cfg, seed=g["seed"]), precision="bf16")
    got = _heads(model, g["arrays"])
    want = g["heads"]
    assert np.isfinite(got).all()
    err = rel_err(got, want)
    assert err < BF16_TOL, f"bf16 heads off by {err:.3e}"
    vt_ref, vt_got = want[:, 2:5], got[:, 2:5]
    srt = np.sort(vt_ref, axis=1)
    confident = (srt[:, -1] - srt[:, -2]) > 2 * BF16_TOL * np.abs(want).max()
    assert np.array_equal(vt_ref.argmax(1)[confident], vt_got.argmax(1)[confident])


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", [min_config(), small_config(pool_combine_dimension=256), min_config(skip_final_maxpool=True)],
                         ids=["min", "small_d256_highway", "min_skip_final_maxpool"])
def test_bf16_matches_fp32_path_at_full_size(cfg):
    err = _bf16_vs_fp32(cfg, 64, seed=3)
    assert err < BF16_TOL, f"bf16 off the fp32 path by {err:.3e}"


@pytest.mark.gpu
def test_bf16_min_fused_and_layerwise_routes_agree():
    cfg = min_config()
    model = build_model(cfg, synth_state_dict(cfg, seed=5), precision="bf16")
    batch = make_pileups(24, seed=51, coverage="poisson")
    fused = _heads(model, batch.arrays())
    layerwise = _heads(model.set_layerwise(True), batch.arrays())
    ref32 = _heads(model.set_layerwise(False).set_precision("fp32"), batch.arrays())
    assert rel_err(layerwise, fused) < BF16_TOL
    assert rel_err(fused, ref32) < BF16_TOL and rel_err(layerwise, ref32) < BF16_TOL


@pytest.mark.gpu
def test_bf16_min_is_batch_shape_invariant():
    """The post-pool GEMM runs K = 51 456 unsplit, so a candidate's heads do not depend on the batch it arrives in: bitwise equal across
    sub-batches, pass sizes and the host-buffer entry point."""
    cfg = min_config()
    model = build_model(cfg, synth_state_dict(cfg, seed=7), precision="bf16")
    batch = make_pileups(40, seed=71, coverage="poisson")
    full = _heads(model, batch.arrays())
    parts = np.concatenate([_heads(model, batch.slice(lo, hi).arrays()) for lo, hi in ((0, 13), (13, 14), (14, 40))])
    assert np.array_equal(full, parts)
    model.set_pass_candidates(7)
    assert np.array_equal(_heads(model, batch.arrays()), full)
    r, q, s, ref, rm, vm = (t.pin_memory() for t in _tensors(batch.arrays()))
    host = model.forward_heads_host(r, ref, q, s, rm, vm)
    torch.cuda.synchronize()
    assert np.array_equal(host.numpy(), full)


def _fc_input_check(cfg, sd, arrays):
    model = build_model(cfg, sd, precision="bf16")
    _heads(model, arrays)
    fc_in = model.debug_fc_input(len(arrays[0])).cpu().numpy()
    r, q, s, ref, rm, vm = arrays
    want = dan_oracle.forward(cfg, sd, r, ref, q, s, rm, vm, keep=True)["fc_in"]
    assert fc_in.shape == want.shape
    scale = np.abs(want).max()
    D = cfg.pool_combine_dimension
    assert np.abs(fc_in[:, :D] - want[:, :D]).max() < 2e-2 * scale, "relu(post_pool(pooled)) block"
    if cfg.highway:
        assert np.abs(fc_in[:, D:] - want[:, D:]).max() < 2e-2 * scale, "highway block"


@pytest.mark.gpu
def test_bf16_fc_input_matches_oracle_min():
    g = load_golden("min_smallfc")
    _fc_input_check(g["cfg"], synth_state_dict(g["cfg"], seed=g["seed"]), g["arrays"])


@pytest.mark.gpu
def test_bf16_fc_input_matches_oracle_with_highway():
    cfg = small_config(pool_combine_dimension=256)
    _fc_input_check(cfg, synth_state_dict(cfg, seed=11), make_pileups(3, seed=12, coverage="poisson").arrays())


@pytest.mark.gpu
def test_bf16_rejects_a_pool_combine_dimension_the_kernels_do_not_take():
    cfg = min_config(layer_sizes=(64, 32), pool_combine_dimension=48)          # a multiple of 16 (fp32 path) but not of 32
    model = build_model(cfg, synth_state_dict(cfg, seed=1), precision="bf16")
    batch = make_pileups(2, seed=1)
    with pytest.raises(NotImplementedError, match="pool_combine_dimension must be a multiple of 32"):
        _heads(model, batch.arrays())
    assert np.isfinite(_heads(model.set_precision("fp32"), batch.arrays())).all()


# ---------------------------------------------------------------------------------------------------------------- training
_NOT_TRAINED = dan_torch_ref.NOT_TRAINED
_train_reference = dan_torch_ref.train_reference


def _sampled(a):
    a = np.asarray(a, np.float64)
    return a.reshape(-1)[::SAMPLE_STRIDE] if a.size > SAMPLE_ABOVE else a


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", [min_config(layer_sizes=(64, 32), pool_combine_dimension=96), small_config(pool_combine_dimension=96, hidden_dropout=0.0)],
                         ids=["min", "small_highway_bn"])
def test_training_step_matches_float64_autograd(cfg):
    sd = synth_state_dict(cfg, seed=21)
    batch = make_pileups(4, seed=22, coverage="poisson")
    cw = np.random.default_rng(23).standard_normal((4, 27)).astype(np.float32)
    dev = torch.device("cuda", 0)
    # reference: float64 autograd (the truth), and fp32 for the error the reference's own precision makes (TF32 off)
    ref = {}
    tf32 = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        for dtype in (torch.float64, torch.float32):
            heads, params, bufs = _train_reference(cfg, sd, batch.arrays(), dtype, dev)
            (heads * torch.from_numpy(cw).to(dev, dtype)).sum().backward()
            grads = {k: v.grad.cpu().numpy() for k, v in params.items() if v.grad is not None}      # BatchNorm off: its parameters are unused
            ref[dtype] = (heads.detach().cpu().numpy(), grads, {k: v.cpu().numpy() for k, v in bufs.items()})
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = tf32
    want_heads, want_grads, want_bufs = ref[torch.float64]

    model = build_model(cfg, sd, precision="fp32").train()
    r, q, s, rf, rm, vm = (t.long() for t in _tensors(batch.arrays()))
    dummy = torch.zeros(4, dtype=torch.long)
    out = model(r, rf, q, s, dummy, dummy, dummy, dummy, rm, vm)
    heads = torch.cat([o.reshape(o.shape[0], -1) for o in out[:6]], dim=1)
    (heads * torch.from_numpy(cw).to(heads.device)).sum().backward()
    assert rel_err(heads.detach().cpu().numpy(), want_heads) < 1e-4, "training-mode forward"

    errs, own = {}, {}
    for name, p in model.named_parameters():
        if name not in want_grads:
            assert p.grad is None or name in _NOT_TRAINED, name
            continue
        assert p.grad is not None, f"no gradient for {name}"
        got, want = _sampled(p.grad.detach().cpu().numpy()), _sampled(want_grads[name])
        scale = max(np.abs(want).max(), 1e-20)
        errs[name] = float(np.abs(got - want).max() / scale)
        own[name] = float(np.abs(_sampled(ref[torch.float32][1][name]) - want).max() / scale)
    assert {"post_pool_conv1D.weight", "post_pool_conv1D.bias"} <= set(errs)
    assert len(errs) == len(want_grads)
    print("gradient error vs float64 autograd, ours | fp32 autograd:", {k: f"{errs[k]:.1e} | {own[k]:.1e}" for k in errs})
    # A few conv-stack tensors are ill-conditioned: their gradients are sums over 80 400 rows that cancel, and the reference's own fp32 run
    # can miss the bar against float64 (PROD topology, batch 4: bottleneck layer 5 weight at 7.3e-3). There the bar is 1.5x what fp32
    # autograd itself achieves.
    bad = {k: (v, own[k]) for k, v in errs.items() if not v < max(GRAD_TOL, 1.5 * own[k])}
    assert not bad, f"gradients off: {bad}"
    for name, b in model.named_buffers():
        if "running_" in name:
            np.testing.assert_allclose(b.detach().cpu().numpy(), want_bufs[name], rtol=2e-5, atol=1e-6, err_msg=name)


@pytest.mark.gpu
def test_training_with_dropout_and_read_removal_is_reproducible():
    cfg = small_config(pool_combine_dimension=96)          # hidden_dropout 0.1; read removal needs the ref / var masks
    sd = synth_state_dict(cfg, seed=9)
    batch = make_pileups(4, seed=17, coverage="poisson")
    r, q, s, ref, rm, vm = (t.long() for t in _tensors(batch.arrays()))
    dummy = torch.zeros(4, dtype=torch.long)

    def run(seed):
        model = build_model(cfg, sd, precision="fp32").train()
        torch.manual_seed(seed)
        out = model(r, ref, q, s, dummy, dummy, dummy, dummy, rm, vm, rm_non_var_reads=1, rm_var_reads=1)
        (out[0].sum() + out[1].pow(2).sum()).backward()
        pp = model.post_pool_conv1D
        return [torch.cat(out[:2], dim=1).detach().cpu().numpy(), pp.weight.grad.cpu().numpy(), pp.bias.grad.cpu().numpy(),
                model.conv1D_layers[3].weight.grad.cpu().numpy()]

    a, b, c = run(1), run(1), run(2)
    assert all(np.array_equal(x, y) for x, y in zip(a, b))
    assert not np.array_equal(a[0], c[0]) and not np.array_equal(a[1], c[1])
    assert np.isfinite(a[1]).all() and np.abs(a[1]).max() > 0


# ---------------------------------------------------------------------------------------------------------------- data parallel (CPU)
def test_post_pool_gradients_go_in_the_first_allreduce_bucket():
    from dl4vc_b200.model import Basic2DNet
    from dl4vc_b200.train_dp import GradientAllReducer
    model = Basic2DNet(**ctor_kwargs(min_config(layer_sizes=(64, 32), pool_combine_dimension=64)))
    first, rest = GradientAllReducer(model).buckets
    pp = model.post_pool_conv1D
    assert any(p is pp.weight for p in first) and any(p is pp.bias for p in first)
    assert not any(p is pp.weight or p is pp.bias for p in rest)
