"""CPU: the oracle (numpy restatement) against goldens produced by the REAL reference (oracle/make_goldens.py)."""
import hashlib

import numpy as np
import pytest

from conftest import rel_err
from dl4vc_b200.weights import synth_state_dict
from oracle import dan_oracle


def test_oracle_matches_reference_goldens(golden):
    cfg = golden["cfg"]
    sd = synth_state_dict(cfg, seed=golden["seed"], as_torch=False)
    reads, q, s, ref, rm, vm = golden["arrays"]
    res = dan_oracle.forward(cfg, sd, reads, ref, q, s, rm, vm, keep=True)
    # integer / encoding work: bit-exact (SHA-256 of the fp32 conv-1 input tensor of the real reference)
    digest = np.frombuffer(hashlib.sha256(np.ascontiguousarray(res["x0"]).tobytes()).digest(), dtype=np.uint8)
    assert np.array_equal(digest, golden["x0_sha256"])
    assert np.array_equal(res["x0"][0][:, [0, 1, cfg.num_reads // 2, cfg.num_reads - 1], :], golden["x0_cand0_reads"])
    # fp32 heads: 1e-4 relative is the product tolerance; the oracle itself sits at ~1e-6
    assert res["heads"].shape == golden["heads"].shape
    assert rel_err(res["heads"], golden["heads"]) < 5e-6
    # per-layer activations of candidate 0
    pool = None
    for l, h in enumerate(res["layers"]):
        a = h[0]
        if golden["layer_includes_pool"][l]:
            a = a + a.mean(axis=1, keepdims=True)
        np.testing.assert_allclose(a[::16, ::33, ::20], golden["layer_sample"][l], rtol=2e-4, atol=5e-5)   # fp32 summation order (up to 300 reads in the pool mean)
        np.testing.assert_allclose(np.abs(a).mean(axis=(1, 2)), golden["layer_absmean"][l], rtol=1e-4, atol=1e-6)
    if cfg.highway:
        hw = np.stack([x[0].reshape(cfg.bottleneck, cfg.num_reads) for x in res["highway"]])
        np.testing.assert_allclose(hw, golden["highway_cand0"], rtol=1e-3, atol=2e-4)
    np.testing.assert_allclose(res["fc_in"][0][::37], golden["fc_in_cand0_sample"], rtol=1e-3, atol=1e-4)


def test_match_masks_bit_exact(golden):
    cfg = golden["cfg"]
    if not cfg.use_reads_ref_var_mask:
        pytest.skip("config has no mask channels")
    reads, q, s, ref, rm, vm = golden["arrays"]
    aR, aV, nzR, nzV = dan_oracle.match_masks(reads, rm, vm)
    k = 2 * cfg.embed_dim + int(cfg.use_q_scores) + int(cfg.use_strands)
    got = np.stack([nzR[:, None, :] & aR[:, :, None], nzV[:, None, :] & aV[:, :, None],
                    np.broadcast_to(nzR[:, None, :], (reads.shape[0], cfg.num_reads, cfg.read_len))], axis=1)
    want = golden["x0_mask_channels"][:, k - 2 * cfg.embed_dim:].astype(np.float32)
    assert np.array_equal(got.astype(np.float32), want)


def test_torch_cpu_port_matches_reference_goldens(golden):
    """bench.py's CPU baseline (oracle/dan_torch_cpu.py: the reference's own torch op sequence) gives the reference's results."""
    from oracle import dan_torch_cpu

    cfg = golden["cfg"]
    sd = synth_state_dict(cfg, seed=golden["seed"])
    reads, q, s, ref, rm, vm = golden["arrays"]
    heads = dan_torch_cpu.forward(cfg, sd, reads, ref, q, s, rm, vm).numpy()
    assert rel_err(heads, golden["heads"]) < 5e-6


def test_float64_torch_reference_matches_reference_goldens(golden):
    """oracle/dan_torch_ref.py, the float64 yardstick of the GPU configuration sweep, gives the reference's results: heads and the
    sampled FC input of candidate 0, with its FC-input blocks tiling the whole vector."""
    import torch

    from oracle import dan_torch_ref

    cfg = golden["cfg"]
    sd = synth_state_dict(cfg, seed=golden["seed"])
    res = dan_torch_ref.forward(cfg, sd, golden["arrays"], dtype=torch.float64)
    assert res.heads.dtype == torch.float64
    assert rel_err(res.heads.numpy(), golden["heads"]) < 5e-6
    fc_in = res.fc_in.numpy()
    np.testing.assert_allclose(fc_in[0][::37], golden["fc_in_cand0_sample"], rtol=1e-3, atol=1e-4)
    assert np.array_equal(np.concatenate([b.numpy() for b in res.blocks.values()], axis=1), fc_in)
