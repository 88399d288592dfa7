"""ctypes loader for libytk_b200.so (the C-ABI drop-in boundary, include/yomitoku_b200.h).

There is no CPU fallback: if the CUDA library is missing the import of any device path raises loudly.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libytk_b200.so")
_lib = None

c_void_p = ctypes.c_void_p
c_int = ctypes.c_int
c_ll = ctypes.c_longlong
c_float_p = ctypes.c_void_p


class YtkError(RuntimeError):
    pass


def _declare(lib):
    lib.ytk_last_error.restype = ctypes.c_char_p
    lib.ytk_last_error.argtypes = []
    lib.ytk_version.restype = c_int
    lib.ytk_launch_count.restype = c_ll
    lib.ytk_gemm_profile_begin.restype = None
    lib.ytk_gemm_profile_end.restype = c_int
    lib.ytk_gemm_profile_end.argtypes = [ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double),
                                         ctypes.POINTER(c_ll)]
    lib.ytk_op_conv2d_f16.restype = c_int
    lib.ytk_op_conv2d_f16.argtypes = [c_void_p, c_int, c_int, c_int, c_int, c_ll, c_void_p, c_void_p,
                                       c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int, c_ll,
                                       c_void_p, c_int, c_ll, c_int, c_int, c_void_p]
    lib.ytk_op_linear_f16.restype = c_int
    lib.ytk_op_linear_f16.argtypes = [c_void_p, c_ll, c_int, c_int, c_void_p, c_int, c_void_p, c_void_p, c_int,
                                       c_ll, c_void_p, c_int, c_ll, c_int, c_void_p]
    lib.ytk_op_attention_f16.restype = c_int
    lib.ytk_op_attention_f16.argtypes = [c_void_p, c_ll, c_ll, c_void_p, c_void_p, c_ll, c_ll, c_void_p, c_ll, c_void_p,
                                         c_int, c_int, c_int, c_int, c_int, c_int, c_void_p]
    lib.ytk_op_rt_topk_f32.restype = c_int
    lib.ytk_op_rt_topk_f32.argtypes = [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]


class YtkAttnSeq(ctypes.Structure):
    _fields_ = [("q_off", c_int), ("q_len", c_int), ("o_off", c_int), ("k_len", c_int), ("k_base", c_ll),
                ("kpad", c_int), ("pad_", c_int)]


class YtkTensor(ctypes.Structure):
    _fields_ = [("name", ctypes.c_char_p), ("data", ctypes.c_void_p), ("ndim", c_int), ("shape", c_ll * 4)]


def _declare_dbnet(lib):
    P = ctypes.POINTER
    lib.ytk_dbnet_create.restype = c_int
    lib.ytk_dbnet_create.argtypes = [P(YtkTensor), c_int, c_int, c_int, P(c_void_p)]
    lib.ytk_dbnet_destroy.restype = None
    lib.ytk_dbnet_destroy.argtypes = [c_void_p]
    lib.ytk_dbnet_device.restype = c_int
    lib.ytk_dbnet_device.argtypes = [c_void_p]
    lib.ytk_parseq_device.restype = c_int
    lib.ytk_parseq_device.argtypes = [c_void_p]
    lib.ytk_dbnet_input_size.restype = c_int
    lib.ytk_dbnet_input_size.argtypes = [c_void_p, c_int, c_int, P(c_int), P(c_int)]
    lib.ytk_dbnet_forward_u8.restype = c_int
    lib.ytk_dbnet_forward_u8.argtypes = [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_int, c_void_p]
    lib.ytk_dbnet_forward_f32.restype = c_int
    lib.ytk_dbnet_forward_f32.argtypes = [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_int, c_void_p]
    lib.ytk_dbnet_flops.restype = ctypes.c_double
    lib.ytk_dbnet_flops.argtypes = [c_void_p, c_int, c_int, c_int]
    lib.ytk_dbnet_debug_tensor.restype = c_int
    lib.ytk_dbnet_debug_tensor.argtypes = [c_void_p, c_int, c_int, c_int, ctypes.c_char_p, c_void_p, c_ll, P(c_int)]


class YtkParseqCfg(ctypes.Structure):
    _fields_ = [(n, c_int) for n in (
        "embed_dim", "enc_heads", "enc_depth", "patch_h", "patch_w", "img_h", "img_w", "num_tokens",
        "max_label_length", "dec_heads", "mlp_ratio", "dec_mlp_ratio", "refine_iters", "repetition_stop",
        "rep_period_max", "rep_min_run_p1", "rep_min_repeats", "decode_ar")]


class YtkCrop(ctypes.Structure):
    _fields_ = [("pix_off", c_ll), ("w", c_int), ("wp", c_int), ("tok_off", c_int), ("ntok", c_int),
                ("group", c_int)]


def _declare_parseq(lib):
    P = ctypes.POINTER
    lib.ytk_parseq_create.restype = c_int
    lib.ytk_parseq_create.argtypes = [P(YtkTensor), c_int, P(YtkParseqCfg), P(c_void_p)]
    lib.ytk_parseq_destroy.restype = None
    lib.ytk_parseq_destroy.argtypes = [c_void_p]
    lib.ytk_parseq_set_refine_iters.restype = None
    lib.ytk_parseq_set_refine_iters.argtypes = [c_void_p, c_int]
    lib.ytk_parseq_forward_crops.restype = c_int
    lib.ytk_parseq_forward_crops.argtypes = [c_void_p, c_void_p, c_int, c_ll, P(YtkCrop), c_int, c_int, c_void_p,
                                             c_void_p, c_void_p, c_void_p]
    lib.ytk_parseq_forward_f32.restype = c_int
    lib.ytk_parseq_forward_f32.argtypes = [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_int, c_void_p,
                                           c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]
    lib.ytk_parseq_last_flops.restype = ctypes.c_double
    lib.ytk_parseq_last_flops.argtypes = [c_void_p]
    lib.ytk_parseq_last_steps.restype = c_int
    lib.ytk_parseq_last_steps.argtypes = [c_void_p]
    lib.ytk_parseq_last_phase_ms.restype = None
    lib.ytk_parseq_last_phase_ms.argtypes = [c_void_p, c_void_p]


class YtkDbRun(ctypes.Structure):
    _fields_ = [("root", c_int), ("y", c_int), ("x0", c_int), ("x1", c_int), ("sum", ctypes.c_double)]


def _declare_crops(lib):
    lib.ytk_dbnet_post_front.restype = c_int
    lib.ytk_dbnet_post_front.argtypes = [c_void_p, c_int, c_int, c_int, ctypes.c_float, c_void_p, c_ll, c_void_p, c_int,
                                         c_void_p, c_void_p]
    lib.ytk_extract_crops_u8.restype = c_int
    lib.ytk_extract_crops_u8.argtypes = [c_void_p, c_int, c_int, c_int, c_void_p, c_int, c_void_p, c_ll, c_void_p, c_ll,
                                         c_void_p]
    lib.ytk_halve_pages_u8.restype = c_int
    lib.ytk_halve_pages_u8.argtypes = [c_void_p, c_int, c_int, c_int, c_void_p, c_int, c_int, c_void_p]


def _declare_rtdetr(lib):
    P = ctypes.POINTER
    lib.ytk_rtdetr_create.restype = c_int
    lib.ytk_rtdetr_create.argtypes = [P(YtkTensor), c_int, c_int, c_int, c_int, P(c_void_p)]
    lib.ytk_rtdetr_destroy.restype = None
    lib.ytk_rtdetr_destroy.argtypes = [c_void_p]
    lib.ytk_rtdetr_device.restype = c_int
    lib.ytk_rtdetr_device.argtypes = [c_void_p]
    lib.ytk_rtdetr_forward_f32.restype = c_int
    lib.ytk_rtdetr_forward_f32.argtypes = [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_int, c_void_p]
    lib.ytk_rtdetr_flops.restype = ctypes.c_double
    lib.ytk_rtdetr_flops.argtypes = [c_void_p, c_int]
    lib.ytk_rtdetr_device_bytes.restype = c_ll
    lib.ytk_rtdetr_device_bytes.argtypes = [c_void_p, c_int]
    lib.ytk_rtdetr_debug_tensor.restype = c_int
    lib.ytk_rtdetr_debug_tensor.argtypes = [c_void_p, c_int, ctypes.c_char_p, c_void_p, c_ll, P(c_int)]


def tensor_table(state_dict):
    """state_dict (name -> torch tensor) -> (ctypes array of YtkTensor, keep-alive list). Tensors are converted to
    contiguous host fp32; integer buffers (num_batches_tracked) are skipped."""
    import torch
    keep, rows = [], []
    for name, t in state_dict.items():
        if not torch.is_floating_point(t):
            continue
        t = t.detach().to("cpu", torch.float32).contiguous()
        if t.dim() > 4:
            raise YtkError("tensor %s has rank %d > 4" % (name, t.dim()))
        nb = name.encode()
        keep.append((t, nb))
        shape = (c_ll * 4)(*(list(t.shape) + [1] * (4 - t.dim())))
        rows.append(YtkTensor(nb, t.data_ptr(), t.dim(), shape))
    arr = (YtkTensor * len(rows))(*rows)
    return arr, keep


def lib():
    """Return the loaded library; build it first if the sources are present and it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise YtkError(
            "libytk_b200.so is not built (%s). Run `python -m yomitoku_b200.build` (needs nvcc). "
            "There is no CPU fallback for the device path." % LIB_PATH)
    l = ctypes.CDLL(LIB_PATH)
    _declare(l)
    _declare_dbnet(l)
    _declare_parseq(l)
    _declare_crops(l)
    _declare_rtdetr(l)
    _lib = l
    return l


def check(status):
    if status != 0:
        raise YtkError(lib().ytk_last_error().decode("utf-8", "replace"))


def ptr(t):
    """Device (or host) pointer of a torch tensor / None."""
    return None if t is None else ctypes.c_void_p(t.data_ptr())
