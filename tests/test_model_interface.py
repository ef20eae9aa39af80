"""CPU: the drop-in module keeps the reference's interface — names, shapes, init RNG stream, error behaviour —
and the C-ABI library loads and exports every symbol include/dan_b200.h declares (no compute without a GPU)."""
import ctypes
import hashlib
import json
import os
import re

import pytest
import torch

from dl4vc_b200 import _lib
from dl4vc_b200.config import prod_config, small_config, state_dict_spec
from dl4vc_b200.factory import ctor_kwargs
from dl4vc_b200.model import Basic2DNet
from oracle.interface_configs import CONFIGS

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("name", sorted(CONFIGS))
def test_state_dict_layout_matches_spec(name):
    cfg = CONFIGS[name]
    model = Basic2DNet(**ctor_kwargs(cfg))
    sd = model.state_dict()
    spec = state_dict_spec(cfg)
    assert list(sd.keys()) == [n for n, _, _ in spec]
    for n, shape, _ in spec:
        assert tuple(sd[n].shape) == tuple(shape), n


def test_prod_parameter_count():
    # SURVEY §0.3: 77 733 413 trainable parameters for the shipped configuration
    total = 0
    for n, shape, kind in state_dict_spec(prod_config()):
        if kind == "param":
            k = 1
            for s in shape:
                k *= s
            total += k
    assert total == 77_733_413
    assert prod_config().macs_per_candidate() == 8_059_296_000


@pytest.mark.parametrize("name", sorted(CONFIGS))
def test_same_names_shapes_and_init_as_reference(name):
    """State-dict names and order, shapes, dtypes and the initial values drawn under torch.manual_seed(1) (bitwise, by SHA-256), and the
    named_parameters() order, against tests/golden/init_state.json; a checkpoint of the recorded layout loads unchanged.
    Provenance of the values (the file's "source" field): recorded from this module at commit 68cf6ee, whose initial values this test had
    found bit-identical to the reference dl4vc/model.py when it still compared with a reference checkout directly. oracle/make_init_golden.py
    re-records them from the reference itself."""
    with open(os.path.join(ROOT, "tests", "golden", "init_state.json")) as f:
        want = json.load(f)["configs"][name]
    torch.manual_seed(1)
    mine = Basic2DNet(**ctor_kwargs(CONFIGS[name]))
    sd = mine.state_dict()
    assert list(sd.keys()) == [k for k, _, _, _ in want["state"]]
    for k, shape, dtype, digest in want["state"]:
        assert list(sd[k].shape) == shape and sd[k].dtype == getattr(torch, dtype), k
        assert hashlib.sha256(sd[k].contiguous().numpy().tobytes()).hexdigest() == digest, f"init differs for {k}"
    mine.load_state_dict({k: torch.zeros(shape, dtype=getattr(torch, dtype)) for k, shape, dtype, _ in want["state"]})
    assert [n for n, _ in mine.named_parameters()] == want["parameters"]


def test_unsupported_options_raise_clearly():
    class A:
        use_transformer = True
        transformer_encoder_heads = 2; num_transformer_layers = 1; transformer_feedforward_dim = 8
        final_transformer_dims = 0; transformer_residual = False; transformer_encoder_dropout = 0.1
    with pytest.raises(NotImplementedError, match="use_transformer"):
        Basic2DNet(3, args=A())
    with pytest.raises(NotImplementedError, match="early_loss_layers"):
        Basic2DNet(3, early_loss_layers=[2])
    with pytest.raises(AssertionError):
        Basic2DNet(3, residual_layer_start=1)


def test_cpu_forward_fails_loudly():
    cfg = small_config()
    model = Basic2DNet(**ctor_kwargs(cfg)).eval()
    x = torch.zeros((1, 201, 100), dtype=torch.long)
    v = torch.zeros((1, 201), dtype=torch.long)
    with pytest.raises(RuntimeError, match="CUDA only"):
        model(x, v, x, x, None, None, None, None, v, v)


def test_library_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "dan_b200.h")).read()
    declared = set(re.findall(r"\b(dan_[a-z0-9_]+)\s*\(", header))
    assert declared == set(_lib.EXPORTED_SYMBOLS)
    if not os.path.exists(_lib.LIB_PATH):
        from dl4vc_b200.build import build
        build()
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for sym in sorted(declared):
        assert hasattr(lib, sym), sym
    lib.dan_version.restype = ctypes.c_char_p
    assert b"sm_100a" in lib.dan_version()


def test_config_struct_matches_header_layout():
    c = _lib.make_config_struct(prod_config())
    assert ctypes.sizeof(c) == 4 * (6 + 3 * _lib.DAN_MAX_LAYERS + 6 + 1 + _lib.DAN_MAX_FC + 2)
    assert list(c.dilation)[:7] == [1, 2, 2, 2, 2, 2, 2]
    assert list(c.is_residual)[:7] == [0, 0, 0, 0, 1, 1, 1]
    assert list(c.pool_after)[:7] == [0, 1, 0, 0, 0, 0, 0]
    assert list(c.fc_sizes)[:2] == [1024, 256]


def test_out_of_range_tokens_raise_like_nn_embedding():
    """nn.Embedding raises IndexError on a token outside the table (model.py:450-459); int64 inputs are range-checked before they are
    narrowed to the kernels' uint8 (a silent wrap would index another row)."""
    import torch
    from dl4vc_b200 import _lib
    from dl4vc_b200.model import Basic2DNet

    ok = torch.tensor([[0, 9, 3]], dtype=torch.int64)
    assert Basic2DNet._u8(ok, "cpu", _lib.VOCAB).dtype == torch.uint8
    for bad in (torch.tensor([[0, 10]], dtype=torch.int64), torch.tensor([[-1, 2]], dtype=torch.int64), torch.tensor([[266]], dtype=torch.int64)):
        with pytest.raises(IndexError):
            Basic2DNet._u8(bad, "cpu", _lib.VOCAB)
    assert Basic2DNet._u8(torch.tensor([[200]], dtype=torch.int64), "cpu").item() == 200      # q-scores / strands / masks: plain bytes
