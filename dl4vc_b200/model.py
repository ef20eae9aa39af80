"""Drop-in replacement for the reference's `dl4vc/model.py` (class Basic2DNet, reference dl4vc/model.py:31-961).

Same constructor arguments and defaults (model.py:35-53), same parameter / buffer names, shapes and registration
order (SURVEY App. B) — so reference checkpoints load unchanged, with or without the DataParallel 'module.' prefix
handled by the caller exactly as before (main.py:117-124) — and the same forward signature and 14-tuple result
(model.py:434-436, 959-961). What differs is where the arithmetic runs: forward() hands raw device pointers of the
uint8 pileup tensors and of the packed weights to the hand-written sm_100a kernels behind the C-ABI in
include/dan_b200.h. There is no PyTorch / CPU fallback: without the CUDA library, or on a configuration the kernels
do not cover, forward raises.

Module construction mirrors the reference's order of nn.Module creation so that `torch.manual_seed(s)` followed by
construction yields bit-identical initial parameters (checked in tests/test_model_interface.py).
"""
from __future__ import annotations

import math
import os
import threading
from itertools import chain

import torch
import torch.nn as nn

from . import _lib
from .config import DanConfig, HEAD_NAMES, MAX_READS, SINGLE_READ_LENGTH, VOCAB_SIZE

# module-level constants kept for importers of the reference module (model.py:16-28)
STRAND_ENCODE_FACTOR = 0.5
NONCE = 0.0001
READ_MIDPOINT = 100
READ_MIDPOINT_DISTANCE = 10
COVER_AVERAGE_NORM = 1. / 100.
CONV_CHANNELS = 100
Q_SCORE_SCALE_FACTOR = 1. / 100.
NUM_SINGLE_READS = 100
BOTTLENECK_SIZE = 16
MIN_RESIDUAL_LAYER = 2

_PRECISIONS = {"fp32": _lib.PRECISION_FP32, "bf16": _lib.PRECISION_BF16}


class _Args:
    """Stand-in for the argparse namespace when `args` is omitted: transformer off (arguments.py defaults)."""
    use_transformer = False
    transformer_encoder_heads = 2
    num_transformer_layers = 3
    transformer_feedforward_dim = 64
    final_transformer_dims = 0
    transformer_residual = False
    transformer_encoder_dropout = 0.1


class _DeviceState:
    """Per-device native state: model handle, packed-weight fingerprint, scratch workspace."""

    def __init__(self):
        self.handle = None
        self.fingerprint = None
        self.keepalive = None
        self.workspace = {}


class _DanTrainFunction(torch.autograd.Function):
    """Training-mode forward / backward through dan_train_forward / dan_backward (include/dan_b200.h). The parameter tensors are
    inputs of the Function, so autograd routes the kernel-computed gradients to them (and through nn.DataParallel's broadcast)."""

    @staticmethod
    def forward(ctx, module, u8, removed, dropout_p, seed, *params):
        heads, tape = module._train_forward_native(u8, removed, dropout_p, seed)
        ctx.module, ctx.u8, ctx.removed, ctx.dropout_p, ctx.seed, ctx.tape = module, u8, removed, dropout_p, seed, tape
        ctx.save_for_backward(heads)
        ctx.param_shapes = [None if p is None else tuple(p.shape) for p in params]
        return heads

    @staticmethod
    def backward(ctx, dheads):
        (heads,) = ctx.saved_tensors
        grads = ctx.module._backward_native(ctx.u8, ctx.removed, ctx.dropout_p, ctx.seed, dheads.contiguous().float(), heads, ctx.tape)
        ctx.tape = None
        return (None, None, None, None, None, *grads)


class Basic2DNet(nn.Module):
    check_tokens = False       # range-check device-resident int64 token inputs before narrowing (synchronises); CPU inputs are always checked
    def __init__(self, target_size, layer_sizes=[1024, 256], pre_conv_dropout=0.1, hidden_dropout=0.1,
                 embed_dim=20, pos_embeddings=True, init_conv_channels=CONV_CHANNELS, final_conv_channels=CONV_CHANNELS,
                 ref_concat_at_reads=True, split_ref_reads_groups=False,
                 use_q_scores=False, use_strands=False,
                 use_naive_variant_encoding=False, expand_bases_naive_variant_encoding=True,
                 use_reads_ref_var_mask=True, ref_var_mask_all=False,
                 single_read_len=SINGLE_READ_LENGTH, num_single_reads=NUM_SINGLE_READS,
                 bottleneck_channels=BOTTLENECK_SIZE, bottleneck_linear_outputs=BOTTLENECK_SIZE,
                 append_bottleneck_highway_reads=True, concat_hw_reads=True,
                 reads_sum_concat_at_reads=False,
                 total_conv_layers=5, residual_layer_start=0, conv_kernel_size=3,
                 use_conv_1d=True, conv_1d_pool_append=False, conv_1d_pool_add=True,
                 conv_1d_pool_layers=[2], use_batchnorm=False,
                 early_loss_layers=[], learn_context_early_loss_balance=True,
                 pool_combine_dimension=0, skip_final_maxpool=False,
                 final_layer_dilation=1, middle_layer_dilation=1,
                 append_trust_region=False, append_num_reads=False, append_allele_frequency=False, args={}):
        super().__init__()
        if isinstance(args, dict) and not args:
            args = _Args()
        # ---- options that select branches outside the accelerated path (SURVEY §2 row 1e) -----------------
        unsupported = []
        if getattr(args, "use_transformer", False): unsupported.append("use_transformer (model.py:279-294)")
        if len(early_loss_layers) > 0: unsupported.append("early_loss_layers (model.py:864-900)")
        if reads_sum_concat_at_reads: unsupported.append("reads_sum_concat_at_reads (model.py:474-490)")
        if not ref_concat_at_reads: unsupported.append("ref_concat_at_reads=False (model.py:524-529)")
        if split_ref_reads_groups: unsupported.append("split_ref_reads_groups (model.py:216)")
        if conv_1d_pool_append: unsupported.append("conv_1d_pool_append (model.py:739-740)")
        if conv_kernel_size != 3: unsupported.append("conv_kernel_size != 3")
        if init_conv_channels != final_conv_channels: unsupported.append("init_conv_channels != final_conv_channels")
        if bottleneck_channels != bottleneck_linear_outputs: unsupported.append("bottleneck_channels != bottleneck_linear_outputs")
        if single_read_len != SINGLE_READ_LENGTH: unsupported.append("single_read_len != 201 (dataset.py:114)")
        if unsupported:
            raise NotImplementedError("dl4vc_b200.Basic2DNet: not covered by the B200 kernels: " + "; ".join(unsupported))
        assert use_conv_1d, "Need use_conv_1d as other methods no longer supported."          # model.py:324
        for l in early_loss_layers:
            assert l < total_conv_layers
        if residual_layer_start > 0:
            assert residual_layer_start >= MIN_RESIDUAL_LAYER, \
                "Do not allow residuals starting at conv layer %s" % residual_layer_start    # model.py:209
        assert not append_num_reads, "append_num_reads is deprecated"                          # model.py:347
        assert not append_trust_region, "append_trust_region is deprecated"                    # model.py:351
        assert not (append_allele_frequency and not use_naive_variant_encoding), "append_AF is deprecated"
        assert not use_naive_variant_encoding, "use_naive_variant_encoding is deprecated"      # model.py:360
        if not (conv_1d_pool_append or conv_1d_pool_add) and len(conv_1d_pool_layers) > 0:
            pass  # the reference asserts lazily inside forward (model.py:744); checked there too

        # ---- attributes the reference exposes ---------------------------------------------------------------
        self.init_conv_channels = init_conv_channels
        self.final_conv_channels = final_conv_channels
        self.single_read_len = single_read_len
        self.num_single_reads = num_single_reads
        self.skip_final_maxpool = skip_final_maxpool
        self.pool_combine_dimension = pool_combine_dimension
        self.pos_embeddings = pos_embeddings
        self.ref_concat_at_reads = ref_concat_at_reads
        self.split_ref_reads_groups = split_ref_reads_groups
        self.use_q_scores = use_q_scores
        self.use_strands = use_strands
        self.use_naive_variant_encoding = use_naive_variant_encoding
        self.expand_bases_naive_variant_encoding = expand_bases_naive_variant_encoding
        self.use_reads_ref_var_mask = use_reads_ref_var_mask
        self.bottleneck_channels = bottleneck_channels
        self.bottleneck_linear_outputs = bottleneck_linear_outputs
        self.append_bottleneck_highway_reads = append_bottleneck_highway_reads
        self.concat_hw_reads = concat_hw_reads
        self.reads_sum_concat_at_reads = reads_sum_concat_at_reads
        self.total_conv_layers = total_conv_layers
        self.residual_layer_start = residual_layer_start
        self.early_loss_layers = early_loss_layers
        self.learn_context_early_loss_balance = learn_context_early_loss_balance
        self.use_transformer = False
        self.use_conv_1d = use_conv_1d
        self.conv_kernel_size = conv_kernel_size
        self.conv_1d_pool_append = conv_1d_pool_append
        self.conv_1d_pool_add = conv_1d_pool_add
        self.conv_1d_pool_layers = conv_1d_pool_layers
        self.use_batchnorm = use_batchnorm
        self.append_trust_region = append_trust_region
        self.append_num_reads = append_num_reads
        self.append_AF = append_allele_frequency
        self.vocab_size = VOCAB_SIZE
        self.embed_dim = embed_dim
        self.pre_conv_dropout = pre_conv_dropout
        self.middle_layer_dilation = middle_layer_dilation
        self.final_layer_dilation = final_layer_dilation
        self.dropout = hidden_dropout

        C, L = init_conv_channels, total_conv_layers
        # ---- parameters, in the reference's creation order (RNG parity) ----------------------------------
        self.embeddings = nn.Embedding(VOCAB_SIZE, embed_dim, padding_idx=0, sparse=False, scale_grad_by_freq=True)
        pe = torch.zeros(single_read_len, embed_dim)
        position = torch.arange(0., single_read_len).unsqueeze(1)
        div_term = torch.exp(torch.arange(0., embed_dim, 2) * -(math.log(10000.0) / embed_dim))
        pe[:, 0::2] = torch.sin(position * div_term)
        pe[:, 1::2] = torch.cos(position * div_term)
        self.register_buffer('pe', pe.unsqueeze(0))

        in_ch = 2 * embed_dim + int(use_q_scores) + int(use_strands) + (3 if use_reads_ref_var_mask else 0)
        self.inter_ave_pool1D_layers = nn.ModuleList(
            [nn.AvgPool2d(kernel_size=(MAX_READS, 1), padding=0, ceil_mode=True) for _ in conv_1d_pool_layers])
        convs, bns, botts, comps, ress = [], [], [], [], []
        self.is_residual_layer, self.add_pooling_layer = [], []
        pool_idx = 0
        for l in range(1, L + 1):
            d = 1 if l == 1 else (middle_layer_dilation if l < L else final_layer_dilation)
            convs.append(nn.Conv2d(in_ch if l == 1 else C, C, kernel_size=(1, 3), stride=1, padding=(0, d), dilation=d, bias=True))
            bns.append(nn.BatchNorm2d(C))
            if l in conv_1d_pool_layers:
                self.add_pooling_layer.append(pool_idx); pool_idx += 1
            else:
                self.add_pooling_layer.append(999)
            is_res = residual_layer_start > 0 and l >= residual_layer_start
            if is_res:
                ress.append(nn.Conv2d(C, C, kernel_size=(1, 1)))
            self.is_residual_layer.append(is_res)
            if append_bottleneck_highway_reads:
                botts.append(nn.Conv2d(C, bottleneck_channels, kernel_size=(1, 1)))
                comps.append(nn.Conv2d(bottleneck_channels, bottleneck_linear_outputs, kernel_size=(1, single_read_len)))
        self.conv1D_layers = nn.ModuleList(convs)
        self.bn1D_layers = nn.ModuleList(bns)
        if append_bottleneck_highway_reads:
            self.conv1D_bottleneck_layers = nn.ModuleList(botts)
            self.conv1D_compression_layers = nn.ModuleList(comps)
        if ress:
            self.residual_conv_layers = nn.ModuleList(ress)
        conv_total_out = (1 if skip_final_maxpool else 2) * C * single_read_len
        if not skip_final_maxpool:
            self.maxPool1D = nn.MaxPool2d(kernel_size=(MAX_READS, 1), padding=0, dilation=1, return_indices=False, ceil_mode=True)
        self.avgPool1D = nn.AvgPool2d(kernel_size=(MAX_READS, 1), padding=0, ceil_mode=True)
        if pool_combine_dimension > 0:
            self.post_pool_conv1D = nn.Linear(conv_total_out, pool_combine_dimension)
        if not skip_final_maxpool:
            self.maxPool1DEarly = nn.ModuleList([])
        self.avgPool1DEarly = nn.ModuleList([])
        input_layer_size = pool_combine_dimension if pool_combine_dimension > 0 else conv_total_out
        if append_bottleneck_highway_reads:
            input_layer_size += (L if concat_hw_reads else 1) * bottleneck_linear_outputs * num_single_reads
        self.layer_sizes = [input_layer_size] + list(map(int, layer_sizes))
        self.final_hidden_size = self.layer_sizes[-1]
        self.nonlinearity = nn.ReLU()
        layer_list = []
        if self.dropout:
            layer_list.append(nn.Dropout(p=self.dropout))
        layer_list.extend(chain.from_iterable(
            [nn.Linear(self.layer_sizes[i], self.layer_sizes[i + 1]), self.nonlinearity, nn.Dropout(p=self.dropout)]
            for i in range(len(self.layer_sizes) - 1)))
        self.conv2hidden = nn.Sequential(*layer_list)
        self.conv2hidden_early, self.fcHidden2Bin_early, self.fcHidden2VT_early = [], [], []
        self.fcHidden2BinTarget = nn.Linear(self.final_hidden_size, 2)
        self.fcHidden2VT = nn.Linear(self.final_hidden_size, 3)
        self.fcHidden2AF = nn.Linear(self.final_hidden_size, 1)
        self.fcHidden2Coverage = nn.Linear(self.final_hidden_size, 1)
        self.fcHidden2VB = nn.Linear(self.final_hidden_size, VOCAB_SIZE)
        self.fcHidden2VR = nn.Linear(self.final_hidden_size, VOCAB_SIZE)
        self.bin_output_weights = nn.Parameter(torch.ones(len(early_loss_layers) + 1) * 0.1)
        self.vt_output_weights = nn.Parameter(torch.ones(len(early_loss_layers) + 1) * 0.1)

        # ---- native side -------------------------------------------------------------------------------
        self.dan_config = DanConfig(
            total_conv_layers=L, channels=C, embed_dim=embed_dim, use_q_scores=bool(use_q_scores),
            use_strands=bool(use_strands), use_reads_ref_var_mask=bool(use_reads_ref_var_mask),
            middle_layer_dilation=middle_layer_dilation, final_layer_dilation=final_layer_dilation,
            use_batchnorm=bool(use_batchnorm), residual_layer_start=residual_layer_start,
            conv_1d_pool_layers=tuple(int(x) for x in conv_1d_pool_layers),
            highway=bool(append_bottleneck_highway_reads), bottleneck=bottleneck_channels,
            concat_hw_reads=bool(concat_hw_reads), pool_combine_dimension=pool_combine_dimension,
            skip_final_maxpool=bool(skip_final_maxpool), layer_sizes=tuple(int(x) for x in layer_sizes),
            hidden_dropout=float(hidden_dropout), num_reads=num_single_reads, read_len=single_read_len)
        self.precision = os.environ.get("DL4VC_B200_PRECISION", "bf16")
        self._native = {}                     # device index -> _DeviceState (shared by DataParallel replicas)
        self._native_lock = threading.Lock()
        self._native_owner = True
        self.last_launch_count = 0

    # ------------------------------------------------------------------------------------------------------
    def set_precision(self, precision: str):
        if precision not in _PRECISIONS:
            raise ValueError(f"precision must be one of {sorted(_PRECISIONS)}")
        self.precision = precision
        return self

    def set_pass_candidates(self, n: int):
        """Candidates per internal conv-stack pass (activations of one pass are meant to stay L2-resident)."""
        self._pass_candidates = int(n)
        for st in self._native.values():
            if st.handle:
                _lib.check(_lib.load_library().dan_model_set_pass_candidates(st.handle, int(n)), "set_pass_candidates")
        return self

    def set_layerwise(self, on: bool = True):
        """Test hook: run the bf16 path layer by layer (the route of configurations the fused conv-stack kernel does not take)."""
        self._flags = _lib.FLAG_LAYERWISE if on else 0
        for st in self._native.values():
            if st.handle:
                _lib.check(_lib.load_library().dan_model_set_flags(st.handle, self._flags), "set_flags")
        return self

    def bf16_route(self) -> int:
        """Test hook: the route a bf16 forward takes with the current flags (dan_model_bf16_route): 0 the bf16 path rejects the
        configuration, 1 the fused conv-stack kernel, 2 layer by layer."""
        dev = self._device()
        with torch.cuda.device(dev):
            st = self._state(dev)
            return _lib.check(_lib.load_library().dan_model_bf16_route(st.handle), "dan_model_bf16_route")

    def _device(self) -> torch.device:
        dev = self.embeddings.weight.device
        if dev.type != "cuda":
            raise RuntimeError("dl4vc_b200.Basic2DNet runs on CUDA only (sm_100a kernels, no CPU path): call .cuda() first "
                               "— the reference does the same unconditionally (main.py:117, model.py:459)")
        return dev

    def _fingerprint(self):
        """Identity + version of every parameter / buffer of the module that OWNS them. nn.DataParallel replicas (main.py:117) hold
        freshly broadcast copies whose data_ptr / _version say nothing about the values, so a replica uses the fingerprint its owner
        took when the replica was made (_replicate_for_data_parallel runs on the owner at every forward)."""
        if not self.__dict__.get("_native_owner", True):
            return self._owner_fingerprint
        return tuple((t.data_ptr(), t._version) for t in chain(self.parameters(), self.buffers()))

    def _state(self, dev: torch.device) -> _DeviceState:
        lib = _lib.load_library()
        with self._native_lock:
            st = self._native.get(dev.index)
            if st is None:
                st = self._native[dev.index] = _DeviceState()
            if st.handle is None:
                h = _lib.C.c_void_p()
                cfg_c = _lib.make_config_struct(self.dan_config)
                _lib.check(lib.dan_model_create(_lib.C.byref(cfg_c), _lib.C.byref(h)), "dan_model_create")
                st.handle = h
                if getattr(self, "_pass_candidates", None):
                    _lib.check(lib.dan_model_set_pass_candidates(h, self._pass_candidates), "set_pass_candidates")
                if getattr(self, "_flags", 0):
                    _lib.check(lib.dan_model_set_flags(h, self._flags), "set_flags")
            fp = self._fingerprint()
            if st.fingerprint != fp:
                self._pack(st, dev)
                st.fingerprint = fp
        return st

    def _pack(self, st: _DeviceState, dev: torch.device):
        """Hand the fp32 parameter tensors to dan_model_load_weights (re-layout + BN folding happen on device)."""
        lib = _lib.load_library()
        w = _lib.DanWeightsC()
        keep = []

        def ptr(t):
            t = t.detach().to(device=dev, dtype=torch.float32).contiguous()
            keep.append(t)
            return t.data_ptr()

        cfg = self.dan_config
        w.embeddings = ptr(self.embeddings.weight)
        w.pe = ptr(self.pe[0] if self.pos_embeddings else torch.zeros_like(self.pe[0]))
        res_i = 0
        for l in range(cfg.total_conv_layers):
            w.conv_w[l] = ptr(self.conv1D_layers[l].weight); w.conv_b[l] = ptr(self.conv1D_layers[l].bias)
            bn = self.bn1D_layers[l]
            w.bn_w[l] = ptr(bn.weight); w.bn_b[l] = ptr(bn.bias)
            w.bn_mean[l] = ptr(bn.running_mean); w.bn_var[l] = ptr(bn.running_var)
            if self.is_residual_layer[l]:
                rc = self.residual_conv_layers[res_i]; res_i += 1
                w.res_w[l] = ptr(rc.weight); w.res_b[l] = ptr(rc.bias)
            if cfg.highway:
                w.bott_w[l] = ptr(self.conv1D_bottleneck_layers[l].weight); w.bott_b[l] = ptr(self.conv1D_bottleneck_layers[l].bias)
                w.comp_w[l] = ptr(self.conv1D_compression_layers[l].weight); w.comp_b[l] = ptr(self.conv1D_compression_layers[l].bias)
        if cfg.pool_combine_dimension > 0:
            w.post_pool_w = ptr(self.post_pool_conv1D.weight); w.post_pool_b = ptr(self.post_pool_conv1D.bias)
        for i, idx in enumerate(cfg.fc_indices):
            w.fc_w[i] = ptr(self.conv2hidden[idx].weight); w.fc_b[i] = ptr(self.conv2hidden[idx].bias)
        heads = [getattr(self, n) for n in HEAD_NAMES]
        w.head_w = ptr(torch.cat([h.weight.detach() for h in heads], dim=0))
        w.head_b = ptr(torch.cat([h.bias.detach() for h in heads], dim=0))
        stream = torch.cuda.current_stream(dev).cuda_stream
        _lib.check(lib.dan_model_load_weights(st.handle, _lib.C.byref(w), stream), "dan_model_load_weights")
        st.keepalive = keep      # released on the next pack; same-stream ordering makes earlier reuse safe

    def _workspace(self, st: _DeviceState, dev, batch: int, prec: int, host: bool = False):
        lib = _lib.load_library()
        need = (lib.dan_workspace_bytes_host if host else lib.dan_workspace_bytes)(st.handle, batch, prec)
        if need == 0:
            raise NotImplementedError("precision '%s' is not available for this configuration: %s"
                                      % (self.precision, lib.dan_last_error().decode(errors="replace")))
        key = (prec, host)
        ws = st.workspace.get(key)
        if ws is None or ws.numel() < need:
            ws = st.workspace[key] = torch.empty(int(need), dtype=torch.uint8, device=dev)
        return ws

    @staticmethod
    def _u8(t, dev, vocab=0):
        """vocab > 0: `t` holds embedding tokens. nn.Embedding raises on a token outside [0, vocab) (model.py:450-459); the kernels
        clamp instead of faulting, so wider-than-uint8 inputs are range-checked before they are narrowed — always for CPU tensors, for
        device tensors only with Basic2DNet.check_tokens (the check synchronises)."""
        if t is None:
            return None
        if t.dtype != torch.uint8:
            if vocab and t.numel() and (t.device.type == "cpu" or Basic2DNet.check_tokens) and (int(t.min()) < 0 or int(t.max()) >= vocab):
                raise IndexError(f"token outside [0, {vocab}) in an embedding input (nn.Embedding would raise 'index out of range in self')")
            t = t.to(torch.uint8)           # narrow on the source device first (the trainer hands int64, trainer.py:520-528)
        return t.to(dev, non_blocking=True).contiguous()

    def forward_heads(self, reads, ref, q_scores=None, strands=None, ref_masks=None, var_masks=None):
        """(B,27) fp32 head matrix [xbinary|xVT|sigmoid(xAF)|leaky_relu(xCov)|xVB|xVR] straight from the kernels."""
        if self.training:
            raise RuntimeError("forward_heads is the eval-mode path (running BatchNorm statistics, no dropout): call .eval() (trainer.py:476) "
                               "or forward_train_heads / forward() under autograd for training")
        dev = self._device()
        lib = _lib.load_library()
        with torch.cuda.device(dev):
            st = self._state(dev)
            prec = _PRECISIONS[self.precision]
            B = int(reads.shape[0])
            P, R = self.single_read_len, self.num_single_reads
            if tuple(reads.shape[1:]) != (P, R):
                raise RuntimeError(f"reads must be (batch, {P}, {R}) [batch, position, read] (dataset.py:672-680), got {tuple(reads.shape)}")
            r8, f8 = self._u8(reads, dev, _lib.VOCAB), self._u8(ref, dev, _lib.VOCAB)
            q8 = self._u8(q_scores, dev) if self.use_q_scores else None
            s8 = self._u8(strands, dev) if self.use_strands else None
            rm8 = self._u8(ref_masks, dev) if self.use_reads_ref_var_mask else None
            vm8 = self._u8(var_masks, dev) if self.use_reads_ref_var_mask else None
            out = torch.empty((B, _lib.NUM_HEAD_OUTPUTS), dtype=torch.float32, device=dev)
            if B == 0:
                return out
            ws = self._workspace(st, dev, B, prec)
            p = lambda t: None if t is None else t.data_ptr()
            stream = torch.cuda.current_stream(dev).cuda_stream
            _lib.check(lib.dan_forward(st.handle, prec, p(r8), p(q8), p(s8), p(f8), p(rm8), p(vm8), B, out.data_ptr(),
                                       ws.data_ptr(), ws.numel(), stream), "dan_forward")
            self.last_launch_count = lib.dan_last_launch_count()
        return out

    def forward_heads_host(self, reads, ref, q_scores=None, strands=None, ref_masks=None, var_masks=None, out=None):
        """Host-buffer variant of forward_heads: uint8 CPU tensors (pinned for true asynchrony) in, (B,27) fp32 CPU tensor out.
        The library cuts the batch into chunks and overlaps the H2D copy of chunk k+1 (side stream) with the kernels of chunk k
        (dan_forward_host). Asynchronous on the current stream: synchronize it before reading `out`."""
        if self.training:
            raise RuntimeError("forward_heads_host is the eval-mode path: call .eval() first")
        dev = self._device()
        lib = _lib.load_library()

        def host_u8(t, used=True, vocab=0):
            if t is None or not used:
                return None
            if t.device.type != "cpu":
                raise RuntimeError("forward_heads_host takes CPU tensors; use forward_heads for device tensors")
            if t.dtype != torch.uint8:
                if vocab and t.numel() and (int(t.min()) < 0 or int(t.max()) >= vocab):
                    raise IndexError(f"token outside [0, {vocab}) in an embedding input (nn.Embedding would raise 'index out of range in self')")
                t = t.to(torch.uint8)
            return t.contiguous()

        with torch.cuda.device(dev):
            st = self._state(dev)
            prec = _PRECISIONS[self.precision]
            B = int(reads.shape[0])
            P, R = self.single_read_len, self.num_single_reads
            if tuple(reads.shape[1:]) != (P, R):
                raise RuntimeError(f"reads must be (batch, {P}, {R}) [batch, position, read] (dataset.py:672-680), got {tuple(reads.shape)}")
            r8, f8 = host_u8(reads, vocab=_lib.VOCAB), host_u8(ref, vocab=_lib.VOCAB)
            q8, s8 = host_u8(q_scores, self.use_q_scores), host_u8(strands, self.use_strands)
            rm8, vm8 = host_u8(ref_masks, self.use_reads_ref_var_mask), host_u8(var_masks, self.use_reads_ref_var_mask)
            if out is None:
                out = torch.empty((B, _lib.NUM_HEAD_OUTPUTS), dtype=torch.float32).pin_memory()
            if B == 0:
                return out
            ws = self._workspace(st, dev, B, prec, host=True)
            p = lambda t: None if t is None else t.data_ptr()
            stream = torch.cuda.current_stream(dev).cuda_stream
            self._host_keepalive = (r8, f8, q8, s8, rm8, vm8, out)          # the copies are asynchronous
            _lib.check(lib.dan_forward_host(st.handle, prec, p(r8), p(q8), p(s8), p(f8), p(rm8), p(vm8), B, out.data_ptr(),
                                            ws.data_ptr(), ws.numel(), stream), "dan_forward_host")
            self.last_launch_count = lib.dan_last_launch_count()
        return out

    # ---- training (dan_train_forward / dan_backward) -------------------------------------------------------
    def _train_params(self):
        """(name, tensor or None) of every tensor that receives a gradient from the kernels, in the order of DanWeightsC."""
        cfg = self.dan_config
        out = [("embeddings", self.embeddings.weight)]
        res_i = 0
        for l in range(cfg.total_conv_layers):
            conv, bn = self.conv1D_layers[l], self.bn1D_layers[l]
            out += [(f"conv_w.{l}", conv.weight), (f"conv_b.{l}", conv.bias)]
            out += [(f"bn_w.{l}", bn.weight if cfg.use_batchnorm else None), (f"bn_b.{l}", bn.bias if cfg.use_batchnorm else None)]
            if self.is_residual_layer[l]:
                rc = self.residual_conv_layers[res_i]; res_i += 1
                out += [(f"res_w.{l}", rc.weight), (f"res_b.{l}", rc.bias)]
            if cfg.highway:
                out += [(f"bott_w.{l}", self.conv1D_bottleneck_layers[l].weight), (f"bott_b.{l}", self.conv1D_bottleneck_layers[l].bias),
                        (f"comp_w.{l}", self.conv1D_compression_layers[l].weight), (f"comp_b.{l}", self.conv1D_compression_layers[l].bias)]
        if cfg.pool_combine_dimension > 0:
            out += [("post_pool_w", self.post_pool_conv1D.weight), ("post_pool_b", self.post_pool_conv1D.bias)]
        for i, idx in enumerate(cfg.fc_indices):
            out += [(f"fc_w.{i}", self.conv2hidden[idx].weight), (f"fc_b.{i}", self.conv2hidden[idx].bias)]
        for n in HEAD_NAMES:
            out += [(f"head_w.{n}", getattr(self, n).weight), (f"head_b.{n}", getattr(self, n).bias)]
        return out

    def _weights_struct(self, tensors: dict, dev, keep: list):
        """name -> tensor (layout of _train_params, heads concatenated as head_w / head_b) into a DanWeightsC of device pointers."""
        w = _lib.DanWeightsC()

        def ptr(t):
            if t is None:
                return None
            t = t.detach()
            if t.device != dev or t.dtype != torch.float32 or not t.is_contiguous():
                t = t.to(device=dev, dtype=torch.float32).contiguous()
            keep.append(t)
            return t.data_ptr()

        for name, t in tensors.items():
            field, _, idx = name.partition(".")
            if field in ("embeddings", "post_pool_w", "post_pool_b", "head_w", "head_b"):
                setattr(w, field, ptr(t))
            else:
                getattr(w, field)[int(idx)] = ptr(t)
        return w

    def _u8_inputs(self, reads, ref, q_scores, strands, ref_masks, var_masks, dev):
        P, R = self.single_read_len, self.num_single_reads
        if tuple(reads.shape[1:]) != (P, R):
            raise RuntimeError(f"reads must be (batch, {P}, {R}) [batch, position, read] (dataset.py:672-680), got {tuple(reads.shape)}")
        return (self._u8(reads, dev, _lib.VOCAB), self._u8(q_scores, dev) if self.use_q_scores else None, self._u8(strands, dev) if self.use_strands else None,
                self._u8(ref, dev, _lib.VOCAB), self._u8(ref_masks, dev) if self.use_reads_ref_var_mask else None,
                self._u8(var_masks, dev) if self.use_reads_ref_var_mask else None)

    def _choose_removed(self, u8, rm_non_var_reads, rm_var_reads):
        """Read-removal augmentation (model.py:633-716): min(rm_var_reads, #eligible) distinct reads per candidate that agree with the
        variant proposal, and min(rm_non_var_reads, #eligible) distinct reads that cover the centre column without agreeing, are replaced
        by the empty-read encoding. The reference draws distinct reads with torch.randperm; here each round draws one read per candidate
        uniformly among its eligible reads that are not yet removed. Returns (B, R) uint8 or None."""
        if not (rm_non_var_reads or rm_var_reads) or not self.use_reads_ref_var_mask:
            return None
        reads, var_masks = u8[0], u8[5]
        nz = (var_masks != 0).unsqueeze(2)
        agree = ((reads * nz) == var_masks.unsqueeze(2)).all(dim=1)                       # (B, R), model.py:607-608
        has_read = reads[:, READ_MIDPOINT, :] != 0
        removed = torch.zeros_like(agree)
        for eligible, rounds in ((agree, int(rm_var_reads)), (has_read & ~agree, int(rm_non_var_reads))):
            for _ in range(rounds):
                eligible = eligible & ~removed
                score = torch.rand(eligible.shape, device=eligible.device).masked_fill(~eligible, -1.0)
                pick = score.argmax(dim=1)
                hit = eligible.any(dim=1)
                removed[torch.arange(len(pick), device=pick.device)[hit], pick[hit]] = True
        return removed.to(torch.uint8).contiguous()

    def _train_forward_native(self, u8, removed, dropout_p, seed):
        dev = self._device()
        lib = _lib.load_library()
        with torch.cuda.device(dev):
            st = self._state(dev)                     # packs the fp32 store from the current parameter values
            B = int(u8[0].shape[0])
            need = lib.dan_train_tape_bytes(st.handle, B)
            if need == 0:
                raise NotImplementedError(lib.dan_last_error().decode(errors="replace"))
            tape = torch.empty(int(need), dtype=torch.uint8, device=dev)
            keep = []
            names = dict(self._train_params())
            heads_w = torch.cat([getattr(self, n).weight.detach() for n in HEAD_NAMES], dim=0)
            tensors = {k: v for k, v in names.items() if not k.startswith("head_")}
            tensors["head_w"] = heads_w
            w = self._weights_struct(tensors, dev, keep)
            for l in range(self.dan_config.total_conv_layers):       # running statistics: updated in place by the kernels
                bn = self.bn1D_layers[l]
                w.bn_mean[l] = bn.running_mean.data_ptr(); w.bn_var[l] = bn.running_var.data_ptr()
            out = torch.empty((B, _lib.NUM_HEAD_OUTPUTS), dtype=torch.float32, device=dev)
            p = lambda t: None if t is None else t.data_ptr()
            stream = torch.cuda.current_stream(dev).cuda_stream
            _lib.check(lib.dan_train_forward(st.handle, _lib.C.byref(w), p(u8[0]), p(u8[1]), p(u8[2]), p(u8[3]), p(u8[4]), p(u8[5]), p(removed), B,
                                             float(dropout_p), int(seed), out.data_ptr(), tape.data_ptr(), tape.numel(), stream), "dan_train_forward")
            self.last_train_launch_count = lib.dan_last_launch_count()
            if self.dan_config.use_batchnorm:
                for bn in self.bn1D_layers:              # like nn.BatchNorm2d in training mode; also tells the packed-weight cache that buffers moved
                    bn.num_batches_tracked += 1
        return out, tape

    def _backward_native(self, u8, removed, dropout_p, seed, dheads, heads, tape):
        dev = self._device()
        lib = _lib.load_library()
        with torch.cuda.device(dev):
            st = self._native[dev.index]
            B = int(u8[0].shape[0])
            keep = []
            params = self._train_params()
            tensors = {k: v for k, v in params if not k.startswith("head_")}
            tensors["head_w"] = torch.cat([getattr(self, n).weight.detach() for n in HEAD_NAMES], dim=0)
            w = self._weights_struct(tensors, dev, keep)
            for l in range(self.dan_config.total_conv_layers):
                bn = self.bn1D_layers[l]
                w.bn_mean[l] = bn.running_mean.data_ptr(); w.bn_var[l] = bn.running_var.data_ptr()
            grads = {k: (None if v is None else torch.empty_like(v, dtype=torch.float32, device=dev, memory_format=torch.contiguous_format))
                     for k, v in params if not k.startswith("head_")}
            hidden = self.final_hidden_size
            grads["head_w"] = torch.empty((_lib.NUM_HEAD_OUTPUTS, hidden), dtype=torch.float32, device=dev)
            grads["head_b"] = torch.empty((_lib.NUM_HEAD_OUTPUTS,), dtype=torch.float32, device=dev)
            gw = self._weights_struct(grads, dev, keep)
            p = lambda t: None if t is None else t.data_ptr()
            stream = torch.cuda.current_stream(dev).cuda_stream
            _lib.check(lib.dan_backward(st.handle, _lib.C.byref(w), p(u8[0]), p(u8[1]), p(u8[2]), p(u8[3]), p(u8[4]), p(u8[5]), p(removed), B,
                                        float(dropout_p), int(seed), dheads.data_ptr(), heads.data_ptr(), _lib.C.byref(gw), tape.data_ptr(), tape.numel(),
                                        stream), "dan_backward")
            self.last_train_launch_count = getattr(self, "last_train_launch_count", 0) + lib.dan_last_launch_count()
            out, row = [], 0
            for name, t in params:
                if name.startswith("head_w."):
                    n = t.shape[0]; out.append(grads["head_w"][row:row + n]); continue
                if name.startswith("head_b."):
                    n = t.shape[0]; out.append(grads["head_b"][row:row + n]); row += n; continue
                out.append(grads[name])
        return out

    def forward_train_heads(self, reads, ref, q_scores=None, strands=None, ref_masks=None, var_masks=None, rm_non_var_reads=0, rm_var_reads=0):
        """(B,27) head matrix of the training-mode forward, autograd-connected to the parameters through the native backward."""
        dev = self._device()
        u8 = self._u8_inputs(reads, ref, q_scores, strands, ref_masks, var_masks, dev)
        removed = self._choose_removed(u8, rm_non_var_reads, rm_var_reads)
        seed = int(torch.randint(0, 2 ** 62, (1,)).item())
        params = [t for _, t in self._train_params()]
        return _DanTrainFunction.apply(self, u8, removed, float(self.dropout), seed, *params)

    def forward(self, reads, ref, q_scores, strands, binary_trust_vector,
                af_scores, ref_bases, var_bases, ref_masks, var_masks,
                rm_non_var_reads=0, rm_var_reads=0, debug=False):
        if len(self.conv_1d_pool_layers) > 0 and not (self.conv_1d_pool_append or self.conv_1d_pool_add):
            assert False, "Require conv_1d_pool_append or conv_1d_pool_add for appending intermediateAvePool1D"   # model.py:744
        if self.training and torch.is_grad_enabled():
            h = self.forward_train_heads(reads, ref, q_scores, strands, ref_masks, var_masks, rm_non_var_reads, rm_var_reads)
        else:
            if rm_non_var_reads or rm_var_reads:
                raise NotImplementedError("read-removal augmentation (model.py:633-716) belongs to the training-mode forward")
            h = self.forward_heads(reads, ref, q_scores, strands, ref_masks, var_masks)
        xbinary, xVT, xAF, xCov, xVB, xVR = h[:, 0:2], h[:, 2:5], h[:, 5:6], h[:, 6:7], h[:, 7:17], h[:, 17:27]
        return (xbinary, xVT, xAF, xCov, xVB, xVR, [], [],
                self.bin_output_weights, self.vt_output_weights, None, None, None, None)

    # ---- test hooks ---------------------------------------------------------------------------------------
    def encode(self, reads, ref, q_scores=None, strands=None, ref_masks=None, var_masks=None, bf16=False):
        """conv-1 input tensor in the reference's logical order (B, Cin, reads, positions) fp32 (model.py:719). bf16=True: what the fused
        bf16 kernel's encoder prologue builds (bf16 values, widened)."""
        dev = self._device()
        lib = _lib.load_library()
        with torch.cuda.device(dev):
            st = self._state(dev)
            B = int(reads.shape[0])
            out = torch.empty((B, self.dan_config.in_channels, self.num_single_reads, self.single_read_len), dtype=torch.float32, device=dev)
            r8, f8 = self._u8(reads, dev, _lib.VOCAB), self._u8(ref, dev, _lib.VOCAB)
            q8 = self._u8(q_scores, dev) if self.use_q_scores else None
            s8 = self._u8(strands, dev) if self.use_strands else None
            rm8 = self._u8(ref_masks, dev) if self.use_reads_ref_var_mask else None
            vm8 = self._u8(var_masks, dev) if self.use_reads_ref_var_mask else None
            p = lambda t: None if t is None else t.data_ptr()
            fn = lib.dan_encode_bf16 if bf16 else lib.dan_encode
            _lib.check(fn(st.handle, p(r8), p(q8), p(s8), p(f8), p(rm8), p(vm8), B, out.data_ptr(),
                          torch.cuda.current_stream(dev).cuda_stream), "dan_encode")
        return out

    def debug_fc_input(self, batch: int):
        """FC-trunk input rows of the last internal chunk of the previous forward (test hook)."""
        dev = self._device()
        lib = _lib.load_library()
        st = self._state(dev)
        prec = _PRECISIONS[self.precision]
        ws = st.workspace[(prec, False)]
        out = torch.empty((batch, self.layer_sizes[0]), dtype=torch.float32, device=dev)
        n = _lib.check(lib.dan_debug_fc_input(st.handle, prec, batch, ws.data_ptr(), out.data_ptr(),
                                              torch.cuda.current_stream(dev).cuda_stream), "dan_debug_fc_input")
        return out[:n]

    def _replicate_for_data_parallel(self):
        replica = super()._replicate_for_data_parallel()
        replica._native_owner = False        # nn.DataParallel replicas (main.py:117) share, but never free, the handles
        replica._owner_fingerprint = self._fingerprint()
        return replica

    def __getstate__(self):
        d = self.__dict__.copy()
        d["_native"] = {}
        d["_native_lock"] = None
        return d

    def __setstate__(self, d):
        self.__dict__.update(d)
        self._native_owner = True
        self._native = {}
        self._native_lock = threading.Lock()

    def __del__(self):
        try:
            lib = _lib._lib
            if lib is None or not self.__dict__.get("_native_owner", False):
                return
            for st in self._native.values():
                if st.handle:
                    lib.dan_model_destroy(st.handle)
                    st.handle = None
        except Exception:
            pass
