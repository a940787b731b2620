"""ctypes binding of the C-ABI library (include/turboprune_b200.h).

This is the ONLY way the Python host reaches the CUDA kernels; signatures mirror the
header one to one.  There is no CPU fallback: if the library is missing or a call fails
the wrappers raise.
"""
import ctypes
import os
from ctypes import POINTER, c_char_p, c_float, c_int, c_int32, c_int64, c_size_t, c_uint64, c_void_p

from . import build as _build

TP_SCORE_MAG, TP_SCORE_SNIP, TP_SCORE_SYNFLOW = 0, 1, 2
TP_ERR_K_RANGE = -4

_lib = None


class ConvDesc(ctypes.Structure):
    _fields_ = [(n, c_int32) for n in
                ("n", "h", "w", "cin", "cout", "r", "s", "stride_h", "stride_w", "pad_h", "pad_w", "p", "q")]


class StageItem(ctypes.Structure):
    _fields_ = [("w", c_void_p), ("mask", c_void_p), ("wf", c_void_p), ("wd", c_void_p)] + \
               [(n, c_int32) for n in ("cout", "cin", "r", "s", "cin_p", "cout_p", "wf_ld")] + \
               [("kmask_f", c_void_p), ("kmask_d", c_void_p)]


# name -> (restype, argtypes); every symbol the header declares
SIGNATURES = {
    "tp_strerror": (c_char_p, [c_int]),
    "tp_last_cuda_error": (c_char_p, []),
    "tp_abi_version": (c_int, []),
    "tp_device_sm_count": (c_int, []),
    "tp_set_pdl": (c_int, [c_int]),
    "tp_topk_workspace_bytes": (c_size_t, [c_int, c_int64]),
    "tp_topk_threshold_mask": (c_int, [POINTER(c_void_p), POINTER(c_void_p), POINTER(c_void_p), POINTER(c_void_p),
                                       POINTER(c_int64), c_int, c_int64, c_int, c_void_p, c_void_p, c_size_t,
                                       POINTER(c_int64), c_void_p]),
    "tp_topk_enqueue": (c_int, [POINTER(c_void_p), POINTER(c_void_p), POINTER(c_void_p), POINTER(c_void_p),
                                POINTER(c_int64), c_int, c_int64, c_int, c_void_p, c_void_p, c_size_t, c_int, c_void_p]),
    "tp_topk_finish": (c_int, [POINTER(c_void_p), POINTER(c_void_p), POINTER(c_int64), c_int, c_int64, c_int, c_void_p,
                               c_void_p, c_size_t, POINTER(c_int64), c_void_p]),
    "tp_apply_threshold": (c_int, [POINTER(c_void_p), POINTER(c_void_p), POINTER(c_void_p), POINTER(c_void_p),
                                   POINTER(c_int64), c_int, c_int, c_void_p, c_void_p, c_size_t, c_void_p]),
    "tp_count_zeros": (c_int, [POINTER(c_void_p), POINTER(c_int64), c_int, c_void_p, c_void_p, c_size_t, c_void_p]),
    "tp_stage_weights": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_int, c_int, c_void_p, c_int,
                                 c_int, c_void_p, c_void_p, c_void_p]),
    "tp_kblock_mask_words": (c_size_t, [c_int64]),
    "tp_stage_batched_workspace_bytes": (c_size_t, [c_int]),
    "tp_stage_weights_batched": (c_int, [POINTER(StageItem), c_int, c_int, c_void_p, c_size_t, c_void_p, c_size_t, c_void_p]),
    "tp_to_nhwc_bf16": (c_int, [c_void_p, c_int, c_int64, c_int64, c_int64, c_int64, c_int, c_int, c_int, c_int,
                                c_void_p, c_int, c_void_p]),
    "tp_im2col_c8": (c_int, [c_void_p] + [c_int] * 11 + [c_void_p, c_int, c_void_p]),
    "tp_im2col_stem": (c_int, [c_void_p, c_int, c_int64, c_int64, c_int64, c_int64] + [c_int] * 13 + [c_void_p, c_int, c_void_p]),
    "tp_cifar_augment": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "tp_cifar_epoch": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_int,
                               c_void_p, c_void_p, c_int, POINTER(c_float), POINTER(c_float), c_int, c_int, c_int, c_int, c_void_p]),
    "tp_synth_normal": (c_int, [c_void_p, c_int64, c_uint64, c_uint64, c_int, c_void_p]),
    "tp_synth_labels": (c_int, [c_void_p, c_int64, c_int, c_uint64, c_uint64, c_void_p]),
    "tp_conv_workspace_bytes": (c_size_t, [POINTER(ConvDesc), c_int]),
    "tp_conv_fprop": (c_int, [POINTER(ConvDesc), c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "tp_conv_stats_rows": (c_size_t, [POINTER(ConvDesc)]),
    "tp_conv_fprop_stats": (c_int, [POINTER(ConvDesc), c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "tp_conv_dgrad": (c_int, [POINTER(ConvDesc), c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "tp_conv_dgrad_partial_rows": (c_size_t, [POINTER(ConvDesc)]),
    "tp_conv_dgrad_bnrelu": (c_int, [POINTER(ConvDesc), c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                     c_void_p, c_void_p, c_void_p]),
    "tp_bn_backward_ext": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64,
                                   c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "tp_conv_wgrad": (c_int, [POINTER(ConvDesc), c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p,
                              c_size_t, c_void_p]),
    "tp_sgd_momentum": (c_int, [POINTER(c_void_p), POINTER(c_void_p), POINTER(c_void_p), POINTER(c_int64), c_int,
                                c_void_p, c_float, c_float, c_int, c_int, c_void_p, c_size_t, c_void_p]),
    "tp_segtable_workspace_bytes": (c_size_t, [c_int]),
    "tp_p2p_allreduce_mask": (c_int, [POINTER(c_void_p), POINTER(c_void_p), c_int, c_int, c_int64, c_void_p, c_float,
                                      c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "tp_bn_workspace_bytes": (c_size_t, [c_int64, c_int]),
    "tp_bn_forward": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                              c_float, c_float, c_int, c_int, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "tp_bn_forward_ext": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                  c_float, c_float, c_int, c_int, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_size_t, c_void_p]),
    "tp_bn_backward": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p,
                               c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "tp_maxpool_forward": (c_int, [c_void_p, c_void_p, c_void_p] + [c_int] * 9 + [c_void_p]),
    "tp_maxpool_backward": (c_int, [c_void_p, c_void_p, c_void_p] + [c_int] * 9 + [c_void_p]),
    "tp_p2p_allreduce_nvls": (c_int, [POINTER(c_void_p), POINTER(c_void_p), c_void_p, c_int, c_int, c_int64, c_void_p, c_float,
                                      c_void_p, c_int, c_void_p, c_void_p]),
}


def lib_path() -> str:
    return _build.lib_path()


def load(build_if_missing: bool = False):
    """dlopen the in-tree library.  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not os.path.isfile(path):
        if build_if_missing:
            _build.build()
        else:
            raise RuntimeError(
                f"turboprune_b200: CUDA library not built ({path} missing). "
                "Run `python -c 'import __graft_entry__ as g; g.build()'`; there is no CPU fallback.")
    lib = ctypes.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError here == header/library mismatch
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


class TurboPruneError(RuntimeError):
    def __init__(self, code, where):
        lib = load()
        msg = lib.tp_strerror(code).decode()
        detail = lib.tp_last_cuda_error().decode() if code == -3 else ""
        super().__init__(f"{where}: {msg} (code {code}) {detail}".strip())
        self.code = code


def check(code: int, where: str):
    if code != 0:
        raise TurboPruneError(code, where)


def ptr_array(tensors):
    """HOST array of device pointers (None -> NULL array)."""
    if tensors is None:
        return None
    arr = (c_void_p * len(tensors))()
    for i, t in enumerate(tensors):
        arr[i] = t.data_ptr() if t is not None else None
    return arr


def i64_array(vals):
    arr = (c_int64 * len(vals))()
    for i, v in enumerate(vals):
        arr[i] = int(v)
    return arr


def stream_ptr(device=None):
    import torch
    return c_void_p(torch.cuda.current_stream(device).cuda_stream)
