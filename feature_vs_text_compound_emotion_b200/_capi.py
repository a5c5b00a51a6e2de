"""ctypes binding of libcer_b200.so (include/cer_b200.h).

The library is the only compute path: there is no CPU or eager-PyTorch fallback.  ``lib()``
raises if the shared object is missing; every wrapper raises ``CerError`` on a non-zero status.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libcer_b200.so")
CER_MAX_MODALS = 4


class CerError(RuntimeError):
    pass


class IrUnit(C.Structure):
    _fields_ = [("cin", C.c_int32), ("depth", C.c_int32), ("stride", C.c_int32), ("has_proj", C.c_int32),
                ("w1", C.c_void_p), ("bias1", C.c_void_p), ("alpha", C.c_void_p),
                ("w2", C.c_void_p), ("bias2", C.c_void_p)]


class IrSe(C.Structure):
    _fields_ = [("hidden", C.c_int32), ("reserved", C.c_int32), ("fc1", C.c_void_p), ("fc2", C.c_void_p)]


class Ir50Weights(C.Structure):
    _fields_ = [("in_h", C.c_int32), ("in_w", C.c_int32),
                ("stem_w", C.c_void_p), ("stem_bias", C.c_void_p), ("stem_alpha", C.c_void_p),
                ("n_units", C.c_int32), ("units", C.POINTER(IrUnit)),
                ("fc_in", C.c_int32), ("emb_dim", C.c_int32),
                ("fc_w", C.c_void_p), ("fc_bias", C.c_void_p)]


class VggConv(C.Structure):
    _fields_ = [("cin", C.c_int32), ("cout", C.c_int32), ("pool_after", C.c_int32), ("w", C.c_void_p), ("bias", C.c_void_p)]


class VggFc(C.Structure):
    _fields_ = [("in_dim", C.c_int32), ("out_dim", C.c_int32), ("relu", C.c_int32), ("w", C.c_void_p), ("bias", C.c_void_p)]


class VggishWeights(C.Structure):
    _fields_ = [("in_h", C.c_int32), ("in_w", C.c_int32), ("c1", C.c_int32),
                ("conv1_w", C.c_void_p), ("conv1_bias", C.c_void_p),
                ("n_convs", C.c_int32), ("convs", C.POINTER(VggConv)),
                ("n_fcs", C.c_int32), ("fcs", C.POINTER(VggFc)), ("zeros", C.c_void_p)]


class VggishStep(C.Structure):
    _fields_ = [("kind", C.c_int32), ("layer", C.c_int32), ("h", C.c_int32), ("w", C.c_int32), ("c", C.c_int32),
                ("out_fp32", C.c_int32), ("pool_fused", C.c_int32)]


class TcnBlock(C.Structure):
    _fields_ = [("c_in", C.c_int32), ("c_out", C.c_int32), ("kernel_size", C.c_int32), ("dilation", C.c_int32),
                ("w1", C.c_void_p), ("b1", C.c_void_p), ("w2", C.c_void_p), ("b2", C.c_void_p),
                ("wd", C.c_void_p), ("bd", C.c_void_p), ("post_scale", C.c_void_p), ("post_shift", C.c_void_p)]


CER_MAX_TCN_BLOCKS = 6
_F = C.c_void_p


class TrainConv(C.Structure):
    _fields_ = [("g", _F), ("v", _F), ("bias", _F), ("dg", _F), ("dv", _F), ("dbias", _F)]


class TrainBlock(C.Structure):
    _fields_ = [("c_in", C.c_int32), ("c_out", C.c_int32), ("dilation", C.c_int32), ("reserved", C.c_int32),
                ("conv1", TrainConv), ("conv2", TrainConv), ("wd", _F), ("bd", _F), ("dwd", _F), ("dbd", _F)]


class TrainModal(C.Structure):
    _fields_ = [("in_dim", C.c_int32), ("n_blocks", C.c_int32), ("blocks", TrainBlock * CER_MAX_TCN_BLOCKS),
                ("bn_w", _F), ("bn_b", _F), ("dbn_w", _F), ("dbn_b", _F), ("bn_mean", _F), ("bn_var", _F),
                ("wqkv", _F), ("bqkv", _F), ("dwqkv", _F), ("dbqkv", _F)]


class HeadTrainSpec(C.Structure):
    _fields_ = [("n_modals", C.c_int32), ("kernel_size", C.c_int32), ("modal_dim", C.c_int32), ("num_heads", C.c_int32),
                ("n_out", C.c_int32), ("precision", C.c_int32),
                ("p_tcn", C.c_double), ("p_fusion", C.c_double), ("bn_momentum", C.c_double),
                ("modal", TrainModal * CER_MAX_MODALS),
                ("wo", _F), ("bo", _F), ("ln_g", _F), ("ln_b", _F), ("wr", _F), ("br", _F),
                ("dwo", _F), ("dbo", _F), ("dln_g", _F), ("dln_b", _F), ("dwr", _F), ("dbr", _F),
                ("grad_flat", _F), ("grad_count", C.c_int64)]


class FusionWeights(C.Structure):
    _fields_ = [("n_modals", C.c_int32), ("dim", C.c_int32 * CER_MAX_MODALS),
                ("modal_dim", C.c_int32), ("num_heads", C.c_int32), ("n_out", C.c_int32),
                ("wqkv", C.c_void_p * CER_MAX_MODALS), ("bqkv", C.c_void_p * CER_MAX_MODALS),
                ("wo", C.c_void_p), ("bo", C.c_void_p), ("ln_g", C.c_void_p), ("ln_b", C.c_void_p),
                ("wr", C.c_void_p), ("br", C.c_void_p)]


# name -> (restype, argtypes); mirrors include/cer_b200.h one to one
SIGNATURES = {
    "cer_last_error": (C.c_char_p, []),
    "cer_version": (C.c_int, []),
    "cer_check_device": (C.c_int, []),
    "cer_ir50_workspace_bytes": (C.c_size_t, [C.POINTER(Ir50Weights), C.c_int64]),
    "cer_ir50_create": (C.c_int, [C.POINTER(C.c_void_p), C.POINTER(Ir50Weights), C.c_int64, C.c_void_p, C.c_size_t]),
    "cer_ir50_workspace_bytes_se": (C.c_size_t, [C.POINTER(Ir50Weights), C.POINTER(IrSe), C.c_int64]),
    "cer_ir50_create_se": (C.c_int, [C.POINTER(C.c_void_p), C.POINTER(Ir50Weights), C.POINTER(IrSe), C.c_int64, C.c_void_p,
                                     C.c_size_t]),
    "cer_ir50_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "cer_ir50_debug_activation": (C.c_int64, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p]),
    "cer_ir50_op_variant": (C.c_int, [C.c_void_p, C.c_int32, C.c_int64, C.c_char_p, C.c_int32]),
    "cer_ir50_run_ops": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p]),
    "cer_conv_last_variant": (C.c_char_p, []),
    "cer_ir50_launches": (C.c_int64, [C.c_void_p, C.c_int64]),
    "cer_ir50_destroy": (None, [C.c_void_p]),
    "cer_conv_forward": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p,
                                   C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "cer_vggish_workspace_bytes": (C.c_size_t, [C.POINTER(VggishWeights), C.c_int64]),
    "cer_vggish_create": (C.c_int, [C.POINTER(C.c_void_p), C.POINTER(VggishWeights), C.c_int64, C.c_void_p, C.c_size_t]),
    "cer_vggish_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "cer_vggish_launches": (C.c_int64, [C.c_void_p, C.c_int64]),
    "cer_vggish_destroy": (None, [C.c_void_p]),
    "cer_vggish_steps": (C.c_int32, [C.c_void_p, C.POINTER(VggishStep), C.c_int32]),
    "cer_vggish_debug_activation": (C.c_int64, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p]),
    "cer_vggish_op_variant": (C.c_int, [C.c_void_p, C.c_int32, C.c_int64, C.c_char_p, C.c_int32]),
    "cer_tcn_block_workspace_bytes": (C.c_size_t, [C.POINTER(TcnBlock), C.c_int64, C.c_int64]),
    "cer_tcn_block_forward": (C.c_int, [C.POINTER(TcnBlock), C.c_void_p, C.c_void_p, C.c_int64, C.c_int64,
                                        C.c_void_p, C.c_size_t, C.c_void_p]),
    "cer_tcn_block_tc_workspace_bytes": (C.c_size_t, [C.POINTER(TcnBlock), C.c_int64, C.c_int64]),
    "cer_tcn_block_tc_forward": (C.c_int, [C.POINTER(TcnBlock), C.c_void_p, C.c_void_p, C.c_int64, C.c_int64,
                                           C.c_void_p, C.c_size_t, C.c_void_p]),
    "cer_fusion_head_forward": (C.c_int, [C.POINTER(FusionWeights), C.POINTER(C.c_void_p), C.c_int64, C.c_void_p,
                                          C.c_void_p, C.c_void_p]),
    "cer_head_last_variant": (C.c_char_p, []),
    "cer_head_train_workspace_bytes": (C.c_size_t, [C.POINTER(HeadTrainSpec), C.c_int64, C.c_int64]),
    "cer_head_train_create": (C.c_int, [C.POINTER(C.c_void_p), C.POINTER(HeadTrainSpec), C.c_int64, C.c_int64, C.c_void_p,
                                        C.c_size_t]),
    "cer_head_train_forward": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.c_uint32, C.c_void_p, C.c_void_p]),
    "cer_head_train_backward": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.c_void_p, C.c_void_p]),
    "cer_head_train_destroy": (None, [C.c_void_p]),
    "cer_head_train_tcn_forward": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.c_uint32, C.POINTER(C.c_void_p), C.c_void_p]),
    "cer_head_train_tcn_backward": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_void_p]),
    "cer_linear_backward": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                      C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "cer_act_backward": (C.c_int, [C.c_int32, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "cer_leaky_relu_forward": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "cer_softmax_gate_backward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "cer_add_layernorm_backward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_float, C.c_void_p, C.c_void_p,
                                             C.c_void_p, C.c_void_p, C.c_void_p]),
    "cer_bn1d_train_forward": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.c_void_p, C.c_void_p, C.c_float, C.c_void_p]),
    "cer_bn1d_train_backward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                          C.c_void_p, C.c_void_p, C.c_void_p]),
    "cer_sdpa_train_forward": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                         C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]),
    "cer_sdpa_backward": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p,
                                    C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32,
                                    C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]),
    "cer_ce_loss": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "cer_optimizer_step": (C.c_int, [C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_float,
                                     C.c_float, C.c_float, C.c_float, C.c_float, C.c_int32, C.c_int32, C.c_float, C.c_void_p]),
    "cer_preproc_workspace_bytes": (C.c_size_t, []),
    "cer_preproc_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_size_t]),
    "cer_preproc_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "cer_preproc_destroy": (None, [C.c_void_p]),
    "cer_logmel_num_frames": (C.c_int64, [C.c_int64, C.c_int32, C.c_int32]),
    "cer_logmel_forward": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_double,
                                     C.c_void_p, C.c_void_p]),
    "cer_frame_examples": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]),
    "cer_linear_forward": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                     C.c_void_p, C.c_int32, C.c_void_p]),
    "cer_softmax_gate": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p]),
    "cer_sdpa_forward": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                   C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p]),
    "cer_sdpa_tc_forward": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                      C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p]),
    "cer_add_layernorm": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_float,
                                    C.c_void_p, C.c_void_p]),
    "cer_modal_attention_maps": (C.c_int, [C.POINTER(C.c_void_p), C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]),
    "cer_modal_attention_forward": (C.c_int, [C.POINTER(C.c_void_p), C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_void_p,
                                              C.c_void_p]),
    "cer_video_vote": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]),
    "cer_add_inplace": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "cer_tanh_inplace": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p]),
    "cer_stitch_windows": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int64,
                                     C.c_void_p, C.c_void_p]),
    "cer_stream_stage": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p,
                                   C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "cer_stream_gather": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p,
                                    C.c_void_p]),
    "cer_stream_average": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p,
                                     C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "cer_stream_retain": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_int32,
                                    C.c_void_p, C.c_void_p]),
}

# int32 fields of cer_stream_entry, in order
STREAM_ENTRY_FIELDS = ("sid", "slot", "lslot", "start", "t_now", "parity", "active", "reserved")

_lib: Optional[C.CDLL] = None


def lib() -> C.CDLL:
    """Load libcer_b200.so (built by feature_vs_text_compound_emotion_b200.build)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise CerError(f"{LIB_PATH} is missing: run `python -m feature_vs_text_compound_emotion_b200.build` "
                           "(there is no fallback path)")
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def check(status: int, what: str = "") -> int:
    if status < 0:
        msg = lib().cer_last_error()
        raise CerError(f"{what} failed with status {status}: {msg.decode() if msg else ''}")
    return status


def require_gpu() -> None:
    """Fail loudly when the kernels cannot run (no CUDA device / not sm_100)."""
    import torch
    if not torch.cuda.is_available():
        raise CerError("no CUDA device: the B200 kernels have no CPU fallback")
    check(lib().cer_check_device(), "cer_check_device")


def current_stream_ptr(device=None) -> int:
    """Raw handle of torch's current stream on ``device`` (default: the current device).  Engines pass
    their own device: a handle taken from another device's current stream is invalid there."""
    import torch
    return torch.cuda.current_stream(device).cuda_stream
