"""ctypes binding of libdan_b200.so (include/dan_b200.h). No torch types cross this boundary: only raw device
pointers, sizes and the raw CUDA stream handle.

The library is REQUIRED: there is no CPU or PyTorch fallback for the forward path; a missing or unloadable .so raises
at first use (DanLibraryError) instead of silently degrading.
"""
from __future__ import annotations

import ctypes as C
import os

DAN_MAX_LAYERS = 12
DAN_MAX_FC = 4
VOCAB = 10              # DAN_VOCAB: rows of the embedding table (model.py:206)
NUM_HEAD_OUTPUTS = 27
PRECISION_FP32 = 0
PRECISION_BF16 = 1
FLAG_LAYERWISE = 1

LIB_PATH = os.environ.get("DAN_B200_LIB") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "libdan_b200.so")   # override: A/B builds during development

# every symbol include/dan_b200.h declares (checked by tests/test_model_interface.py and __graft_entry__.build)
EXPORTED_SYMBOLS = (
    "dan_last_error", "dan_version", "dan_model_create", "dan_model_destroy", "dan_model_load_weights",
    "dan_model_set_pass_candidates", "dan_workspace_bytes", "dan_forward", "dan_workspace_bytes_host",
    "dan_forward_host", "dan_scores", "dan_genotype_calls", "dan_format_vcf_info", "dan_make_mask_vectors", "dan_encode", "dan_encode_bf16", "dan_model_set_flags", "dan_model_bf16_route", "dan_train_tape_bytes", "dan_train_forward", "dan_backward", "dan_losses", "dan_close_table_update", "dan_decode_records", "dan_decode_record_headers", "dan_record_sidecars", "dan_decode_sidecar_headers", "dan_inflate_device", "dan_deflate_bound", "dan_deflate_device", "dan_deflate_compact", "dan_bgzf_compress_device", "dan_bgzf_compact", "dan_decode_layout", "dan_decode_records_device", "dan_debug_fc_input", "dan_last_launch_count", "dan_measure_fma_tflops",
    "dan_profile_enable", "dan_profile_read", "dan_profile_class_name",
)
PROF_NUM_CLASSES = 4
RECORDS_RAW = 0         # DAN_RECORDS_RAW / DAN_RECORDS_ZLIB: the two record formats of dan_decode_records_device
RECORDS_ZLIB = 1


class DanLibraryError(RuntimeError):
    pass


class DanConfigC(C.Structure):
    _fields_ = [
        ("total_conv_layers", C.c_int32), ("channels", C.c_int32), ("embed_dim", C.c_int32),
        ("use_q_scores", C.c_int32), ("use_strands", C.c_int32), ("use_reads_ref_var_mask", C.c_int32),
        ("dilation", C.c_int32 * DAN_MAX_LAYERS), ("is_residual", C.c_int32 * DAN_MAX_LAYERS),
        ("pool_after", C.c_int32 * DAN_MAX_LAYERS),
        ("use_batchnorm", C.c_int32), ("highway", C.c_int32), ("bottleneck", C.c_int32),
        ("concat_hw_reads", C.c_int32), ("pool_combine_dimension", C.c_int32), ("skip_final_maxpool", C.c_int32),
        ("num_fc", C.c_int32), ("fc_sizes", C.c_int32 * DAN_MAX_FC),
        ("num_reads", C.c_int32), ("read_len", C.c_int32),
    ]


class DanFeederConfigC(C.Structure):
    _fields_ = [("max_reads", C.c_int32), ("store_max_reads", C.c_int32), ("use_q_scores", C.c_int32), ("use_strands", C.c_int32),
                ("keep_candidate_af", C.c_int32), ("seed", C.c_uint64)]


class DanRecordBatchC(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("reads", "q_scores", "strands", "ref", "ref_masks", "var_masks", "label", "num_reads", "is_snp",
                                          "var_type", "allele_freq", "coverage", "var_base_enum", "var_ref_enum", "blacklist", "status")]


class DanStagingLayoutC(C.Structure):
    _fields_ = [(n, C.c_size_t) for n in ("sidecars", "records", "stream_offsets", "stream_lengths", "headers", "ref_masks", "var_masks",
                                          "streams", "staging_bytes", "workspace_bytes")]


_PL = C.c_void_p * DAN_MAX_LAYERS
_PF = C.c_void_p * DAN_MAX_FC


class DanWeightsC(C.Structure):
    _fields_ = [
        ("embeddings", C.c_void_p), ("pe", C.c_void_p),
        ("conv_w", _PL), ("conv_b", _PL), ("bn_w", _PL), ("bn_b", _PL), ("bn_mean", _PL), ("bn_var", _PL),
        ("res_w", _PL), ("res_b", _PL), ("bott_w", _PL), ("bott_b", _PL), ("comp_w", _PL), ("comp_b", _PL),
        ("post_pool_w", C.c_void_p), ("post_pool_b", C.c_void_p),
        ("fc_w", _PF), ("fc_b", _PF), ("head_w", C.c_void_p), ("head_b", C.c_void_p),
    ]


_lib = None


def load_library(path: str | None = None):
    """dlopen the CUDA library (once). Raises DanLibraryError if it is absent — build it with
    `python -m dl4vc_b200.build` (or __graft_entry__.build())."""
    global _lib
    if _lib is not None:
        return _lib
    path = path or LIB_PATH
    if not os.path.exists(path):
        raise DanLibraryError(f"{path} not found: the DAN forward has no fallback path; run `python -m dl4vc_b200.build`")
    try:
        lib = C.CDLL(path)
    except OSError as e:  # pragma: no cover
        raise DanLibraryError(f"cannot load {path}: {e}") from e
    vp, i32, sz = C.c_void_p, C.c_int, C.c_size_t
    lib.dan_last_error.restype = C.c_char_p
    lib.dan_version.restype = C.c_char_p
    lib.dan_model_create.argtypes = [C.POINTER(DanConfigC), C.POINTER(vp)]
    lib.dan_model_destroy.argtypes = [vp]
    lib.dan_model_load_weights.argtypes = [vp, C.POINTER(DanWeightsC), vp]
    lib.dan_model_set_pass_candidates.argtypes = [vp, i32]
    lib.dan_workspace_bytes.argtypes = [vp, i32, i32]
    lib.dan_workspace_bytes.restype = sz
    lib.dan_workspace_bytes_host.argtypes = [vp, i32, i32]
    lib.dan_workspace_bytes_host.restype = sz
    fwd = [vp, i32, vp, vp, vp, vp, vp, vp, i32, vp, vp, sz, vp]
    lib.dan_forward.argtypes = fwd
    lib.dan_forward_host.argtypes = fwd
    lib.dan_encode.argtypes = [vp, vp, vp, vp, vp, vp, vp, i32, vp, vp]
    lib.dan_encode_bf16.argtypes = [vp, vp, vp, vp, vp, vp, vp, i32, vp, vp]
    lib.dan_model_set_flags.argtypes = [vp, i32]
    lib.dan_model_bf16_route.argtypes = [vp]
    lib.dan_train_tape_bytes.argtypes = [vp, i32]
    lib.dan_train_tape_bytes.restype = sz
    lib.dan_train_forward.argtypes = [vp, C.POINTER(DanWeightsC), vp, vp, vp, vp, vp, vp, vp, i32, C.c_float, C.c_uint64, vp, vp, sz, vp]
    lib.dan_backward.argtypes = [vp, C.POINTER(DanWeightsC), vp, vp, vp, vp, vp, vp, vp, i32, C.c_float, C.c_uint64, vp, vp, C.POINTER(DanWeightsC), vp, sz, vp]
    lib.dan_debug_fc_input.argtypes = [vp, i32, i32, vp, vp, vp]
    lib.dan_scores.argtypes = [vp, i32, vp, vp]
    lib.dan_genotype_calls.argtypes = [vp, vp, vp, i32, vp, vp, vp, vp]
    lib.dan_format_vcf_info.argtypes = [vp, i32, vp, sz]
    lib.dan_make_mask_vectors.argtypes = [vp, vp, vp, i32, vp, vp, vp]
    cfgp, batchp = C.POINTER(DanFeederConfigC), C.POINTER(DanRecordBatchC)
    lib.dan_decode_records.argtypes = [vp, sz, vp, i32, cfgp, batchp]
    lib.dan_decode_record_headers.argtypes = [vp, sz, vp, i32, cfgp, batchp, vp]
    lib.dan_record_sidecars.argtypes = [vp, sz, i32, vp]
    lib.dan_decode_sidecar_headers.argtypes = [vp, vp, i32, cfgp, batchp, vp]
    lib.dan_decode_layout.argtypes = [i32, i32, sz, C.POINTER(DanStagingLayoutC)]
    lib.dan_decode_records_device.argtypes = [i32, vp, sz, vp, i32, cfgp, batchp, vp, sz, vp, vp]
    lib.dan_inflate_device.argtypes = [vp, vp, vp, i32, vp, C.c_uint64, vp, vp]
    lib.dan_deflate_bound.argtypes = [C.c_uint64]
    lib.dan_deflate_bound.restype = sz
    lib.dan_deflate_device.argtypes = [vp, i32, C.c_uint64, vp, vp, vp, vp]
    lib.dan_deflate_compact.argtypes = [vp, vp, i32, C.c_uint64, vp, vp, vp]
    lib.dan_bgzf_compress_device.argtypes = [vp, C.c_uint64, vp, vp, vp, vp]
    lib.dan_bgzf_compact.argtypes = [vp, vp, i32, vp, vp, vp]
    lib.dan_last_launch_count.restype = i32
    lib.dan_measure_fma_tflops.argtypes = [C.c_double, vp]
    lib.dan_measure_fma_tflops.restype = C.c_double
    lib.dan_profile_enable.argtypes = [i32]
    lib.dan_profile_read.argtypes = [C.POINTER(C.c_double), C.POINTER(C.c_int), i32]
    lib.dan_profile_class_name.argtypes = [i32]
    lib.dan_profile_class_name.restype = C.c_char_p
    _lib = lib
    return lib


def check(rc: int, what: str):
    if rc < 0:
        msg = load_library().dan_last_error().decode(errors="replace")
        if rc == -2:
            raise NotImplementedError(f"{what}: {msg}")
        raise RuntimeError(f"{what} failed ({rc}): {msg}")
    return rc


def make_config_struct(cfg) -> DanConfigC:
    """dl4vc_b200.config.DanConfig -> dan_config."""
    c = DanConfigC()
    L = cfg.total_conv_layers
    if L > DAN_MAX_LAYERS:
        raise NotImplementedError(f"at most {DAN_MAX_LAYERS} conv layers")
    if len(cfg.layer_sizes) > DAN_MAX_FC:
        raise NotImplementedError(f"at most {DAN_MAX_FC} FC layers")
    c.total_conv_layers, c.channels, c.embed_dim = L, cfg.channels, cfg.embed_dim
    c.use_q_scores, c.use_strands = int(cfg.use_q_scores), int(cfg.use_strands)
    c.use_reads_ref_var_mask = int(cfg.use_reads_ref_var_mask)
    for l in range(1, L + 1):
        c.dilation[l - 1] = cfg.dilation(l)
        c.is_residual[l - 1] = int(cfg.is_residual(l))
        c.pool_after[l - 1] = int(l in cfg.conv_1d_pool_layers)
    c.use_batchnorm, c.highway, c.bottleneck = int(cfg.use_batchnorm), int(cfg.highway), cfg.bottleneck
    c.concat_hw_reads, c.pool_combine_dimension = int(cfg.concat_hw_reads), cfg.pool_combine_dimension
    c.skip_final_maxpool = int(cfg.skip_final_maxpool)
    c.num_fc = len(cfg.layer_sizes)
    for i, n in enumerate(cfg.layer_sizes):
        c.fc_sizes[i] = int(n)
    c.num_reads, c.read_len = cfg.num_reads, cfg.read_len
    return c
