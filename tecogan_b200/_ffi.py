"""ctypes binding of libteco.so (include/teco.h).  PyTorch tensors are only the buffer currency:
every call passes raw device pointers, sizes and the current CUDA stream.

No CPU fallback: if the shared library is missing this module raises at import of the first
symbol; if a tensor is not a contiguous CUDA tensor of the expected dtype the wrappers raise.
"""
import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("TECO_LIB", os.path.join(_HERE, "libteco.so"))   # TECO_LIB: A/B-test another build of the same ABI

ACT_NONE, ACT_RELU, ACT_LRELU02, ACT_TANH24, ACT_SIGMOID = 0, 1, 2, 3, 4


class ConvDesc(C.Structure):
    """struct teco_conv_desc (include/teco.h)."""
    _fields_ = [(n, C.c_int32) for n in (
        "N", "H", "W", "Cin", "OH", "OW", "Cout", "KH", "KW", "stride", "pad_t", "pad_l", "out_H", "out_W",
        "out_sy", "out_oy", "out_sx", "out_ox", "in_cpitch", "out_cpitch", "act")] + [
        ("post_scale", C.c_float), ("post_shift", C.c_float)]


class TcDesc(C.Structure):
    """struct teco_tc_desc (include/teco.h)."""
    _fields_ = [(n, C.c_int32) for n in ("N", "H", "W", "Cin", "Cout", "act", "mode", "out_f32_c")] + [
        ("post_scale", C.c_float), ("post_shift", C.c_float)]


_P, _I32, _I64, _F, _D = C.c_void_p, C.c_int32, C.c_int64, C.c_float, C.c_double

# symbol -> argtypes (restype is int unless listed in _RESTYPES).  Mirrors include/teco.h one to one;
# tests/test_abi.py checks this table against the header and against the built library.
SIGNATURES = {
    "teco_version": [],
    "teco_device_props": [C.c_int, _P],
    "teco_crc32c": [_P, _I64, _I64],
    "teco_conv2d_f32": [C.POINTER(ConvDesc), _P, _P, _P, _P, _P, _P],
    "teco_conv2d_wgrad_f32": [C.POINTER(ConvDesc), _P, _P, _P, _P, C.c_int, _P],
    "teco_pack_conv3x3_bf16": [_P, _I32, _I32, _I32, _I32, _I32, _P, _P, _P],
    "teco_packed_weight_bytes": [_I32, _I32],
    "teco_conv3x3_tc": [C.POINTER(TcDesc), _P, _P, _P, _P, _P, _P, _P, _P],
    "teco_bias_grad_f32": [_P, _P, _I64, _I32, _I32, _I32, _P],
    "teco_conv3x3_wgrad_tc": [_I32, _I32, _I32, _I32, _I32, _I32, _I32, _P, _P, _P, _I32, _P],
    "teco_debug_timing": [_P],
    "teco_conv3x3_lin_supported": [_I32, _I32, _I32, _I32],
    "teco_conv3x3_lin_tc": [_I32, _I32, _I32, _I32, _P, _P, _P, _P, _P, _P, _P],
    "teco_warp_f32": [_P, _P, _P, _I32, _I32, _I32, _I32, _P],
    "teco_warp_bwd_f32": [_P, _P, _P, _P, _P, _I32, _I32, _I32, _I32, _P],
    "teco_warp_s2d_fused": [_P, _P, _P, _P, _I32, _I32, _I32, _I32, _I32, _I32, _I32, _I32, _F, _F, _P],
    "teco_upscale4_f32": [_P, _P, _I32, _I32, _I32, _I32, _F, _P],
    "teco_bicubic4_f32": [_P, _P, _I32, _I32, _I32, _I32, _I32, _P],
    "teco_resize_bilinear_f32": [_P, _P, _I32, _I32, _I32, _I32, _I32, _I32, _P],
    "teco_resize_bilinear_bwd_f32": [_P, _P, _I32, _I32, _I32, _I32, _I32, _I32, _P],
    "teco_maxpool2_f32": [_P, _P, _I32, _I32, _I32, _I32, _P],
    "teco_maxpool2_bwd_f32": [_P, _P, _P, _I32, _I32, _I32, _I32, _P],
    "teco_maxpool2_bf16": [_P, _P, _I32, _I32, _I32, _I32, _P],
    "teco_resize2x_bf16": [_P, _P, _I32, _I32, _I32, _I32, _P],
    "teco_space_to_depth4_f32": [_P, _P, _I32, _I32, _I32, _I32, _I32, _I32, _P],
    "teco_depth_to_space4_f32": [_P, _P, _I32, _I32, _I32, _I32, _I32, _I32, _P],
    "teco_gauss_down4_f32": [_P, _P, _I32, _I32, _I32, _I32, _P],
    "teco_affine_act_f32": [_P, _P, _I64, _F, _F, _I32, _P],
    "teco_act_bwd_f32": [_P, _P, _P, _I64, _I32, _P],
    "teco_f32_to_bf16_pad": [_P, _P, _I64, _I32, _I32, _I32, _I32, _F, _F, _P],
    "teco_bf16_to_f32": [_P, _P, _I64, _I32, _I32, _I32, _P],
    "teco_bf16_to_f32_add": [_P, _P, _P, _I64, _I32, _I32, _I32, _P],
    "teco_f32_to_bf16_rowpad": [_P, _P, _I64, _I32, _I32, _I32, _P],
    "teco_to_u8": [_P, _P, _I64, _P],
    "teco_deprocess_u8": [_P, _P, _P, _I64, _P],
    "teco_bn_train_f32": [_P, _P, _P, _P, _I64, _I32, _F, _I32, _P],
    "teco_bn_train_bwd_f32": [_P, _P, _P, _P, _P, _P, _I64, _I32, _F, _I32, _P],
    "teco_loss_l2_f32": [_P, _P, _P, _P, _I64, _I32, _F, _P],
    "teco_loss_l1_f32": [_P, _P, _P, _P, _P, _I64, _I32, _I32, _F, _P],
    "teco_loss_cosine_f32": [_P, _P, _P, _P, _I64, _I32, _F, _P],
    "teco_l2norm_channels_f32": [_P, _P, _I64, _I32, _P],
    "teco_loss_gan_f32": [_P, _P, _P, _P, _P, _P, _I64, _F, _F, _F, _P],
    "teco_adam_f32": [_P, _P, _P, _P, _I64, _F, _F, _F, _F, _F, _P],
    "teco_metrics_psnr_y_u8": [_P, _I32, _I32, _P, _I32, _I32, _I32, _I32, _I32, _I32, _I32, _P, _P],
    "teco_metrics_ssim_y_u8": [_P, _I32, _I32, _P, _I32, _I32, _I32, _I32, _I32, _I32, _I32, _P, _P],
    "teco_grey_u8": [_P, _I32, _I32, _I32, _I32, _I32, _P, _P],
    "teco_farneback_workspace_bytes": [_I32, _I32, _I32, _I32, _D, _I32],
    "teco_farneback_flow": [_P, _I32, _I32, _I32, _P, _I32, _D, _I32, _I32, _I32, _I32, _D, _I32, _P, _I64, _P, _P],
    "teco_tof_sums": [_P, _P, _I32, _I32, _I32, _I32, _I32, _I32, _I32, _P, _P],
}
_RESTYPES = {"teco_packed_weight_bytes": C.c_int64, "teco_crc32c": C.c_int64, "teco_farneback_workspace_bytes": C.c_int64}

_lib = None


def lib():
    """Load libteco.so once.  Fails loudly: there is no other implementation to fall back to."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "tecogan_b200: %s not found -- build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a).  There is no CPU or PyTorch fallback." % LIB_PATH)
        l = C.CDLL(LIB_PATH)
        for name, args in SIGNATURES.items():
            fn = getattr(l, name)
            fn.argtypes = args
            fn.restype = _RESTYPES.get(name, C.c_int)
        l.teco_last_error.argtypes = []
        l.teco_last_error.restype = C.c_char_p
        _lib = l
    return _lib


def check(rc):
    """Map C-ABI return codes to the reference's exception style: ValueError for misuse
    (lib/frvsr.py:46-47 etc.), RuntimeError for CUDA failures."""
    if rc == 0:
        return
    msg = lib().teco_last_error().decode("utf-8", "replace")
    if rc == -1:
        raise ValueError(msg)
    raise RuntimeError("libteco error %d: %s" % (rc, msg))


def stream_ptr():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t, dtype=None):
    """Device pointer of a contiguous CUDA tensor (None -> NULL)."""
    if t is None:
        return C.c_void_p(0)
    if not t.is_cuda:
        raise ValueError("tecogan_b200 needs CUDA tensors (there is no CPU path); got a %s tensor" % t.device)
    if not t.is_contiguous():
        raise ValueError("tecogan_b200 needs contiguous NHWC tensors")
    if dtype is not None and t.dtype != dtype:
        raise ValueError("expected dtype %s, got %s" % (dtype, t.dtype))
    return C.c_void_p(t.data_ptr())


def call(name, *args):
    check(getattr(lib(), name)(*args))
