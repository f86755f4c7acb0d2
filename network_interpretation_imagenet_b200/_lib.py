"""ctypes binding of libnib.so (include/nib.h).

This is the *only* compute backend: if the shared library is missing, or no sm_100 device is
present when a compute call is made, the call raises.  There is no CPU or PyTorch fallback
(the CPU restatement in `oracle/` is test infrastructure and is never imported from here).
"""
from __future__ import annotations

import ctypes as C
import os

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(PKG_DIR, "libnib.so")

NIB_OK = 0
ABI_VERSION = 4
MASK_KEEP_MUL, MASK_REMOVE_MINMAX = 0, 1
F32, BF16 = 0, 1
NCHW, NHWC = 0, 1
PREC_FP32, PREC_BF16, PREC_X3, PREC_SPLIT = 0, 1, 2, 3
CONV_RELU, CONV_PRE_BNRELU = 1, 2
POOL_MAX, POOL_AVG = 0, 1
IN_NCHW_F32, IN_NATIVE = 0, 1


class NibError(RuntimeError):
    def __init__(self, code: int, where: str, msg: str):
        super().__init__(f"{where} failed with code {code}: {msg}")
        self.code = code


class MaskArgs(C.Structure):
    _fields_ = [
        ("d_img", C.c_void_p), ("d_labels", C.c_void_p), ("label_bytes", C.c_int),
        ("d_sel", C.c_void_p), ("sel_words", C.c_int),
        ("N", C.c_int), ("C", C.c_int), ("H", C.c_int), ("W", C.c_int), ("S", C.c_int),
        ("mode", C.c_int), ("d_seg_minmax", C.c_void_p),
        ("d_out", C.c_void_p), ("out_dtype", C.c_int), ("layout", C.c_int),
        ("c_stride", C.c_int), ("pad_h", C.c_int), ("pad_w", C.c_int),
        ("d_pixel_mask", C.c_void_p),
    ]


class ConvDesc(C.Structure):
    _fields_ = [
        ("in_buf", C.c_int), ("in_coff", C.c_int), ("Cin", C.c_int),
        ("out_buf", C.c_int), ("out_coff", C.c_int), ("Cout", C.c_int),
        ("res_buf", C.c_int), ("res_coff", C.c_int), ("res_C", C.c_int),
        ("R", C.c_int), ("S", C.c_int), ("stride", C.c_int), ("pad", C.c_int),
        ("flags", C.c_int),
    ]


_vp, _i, _d = C.c_void_p, C.c_int, C.c_double
_PROTOTYPES = {
    "nib_abi_version": (C.c_int, []),
    "nib_last_error": (C.c_char_p, []),
    "nib_device_info": (_i, [_i, C.POINTER(_i), C.POINTER(_i), C.POINTER(_i)]),
    "nib_segment_minmax": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _vp, _vp]),
    "nib_mask_synth": (_i, [C.POINTER(MaskArgs), _vp]),
    "nib_mask_display_u8": (_i, [C.POINTER(MaskArgs), _vp, _vp]),
    "nib_prep_minmax_u8": (_i, [_vp, _i, _i, _i, _vp, _vp]),
    "nib_net_create": (_i, [_i, _i, C.POINTER(_vp)]),
    "nib_net_destroy": (_i, [_vp]),
    "nib_net_add_buffer": (_i, [_vp, _i, _i, _i, _i]),
    "nib_net_add_buffer_f32": (_i, [_vp, _i, _i, _i, _i]),
    "nib_net_add_convert": (_i, [_vp, _i, _i]),
    "nib_net_add_conv": (_i, [_vp, C.POINTER(ConvDesc), _vp, _vp, _vp, _vp]),
    "nib_net_add_pool": (_i, [_vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _vp]),
    "nib_net_add_fc": (_i, [_vp, _i, _i, _i, _vp, _vp]),
    "nib_net_set_input": (_i, [_vp, _i]),
    "nib_net_finalize": (_i, [_vp]),
    "nib_net_forward": (_i, [_vp, _vp, _i, _i, _vp, _vp]),
    "nib_net_forward_masked": (_i, [_vp, C.POINTER(MaskArgs), _vp, _vp]),
    "nib_net_buffer_info": (_i, [_vp, _i, C.POINTER(_vp), C.POINTER(_i), C.POINTER(_i), C.POINTER(_i),
                                 C.POINTER(_i), C.POINTER(_i)]),
    "nib_net_read_buffer_nchw": (_i, [_vp, _i, _i, _vp, _vp]),
    "nib_net_launch_counts": (_i, [_vp, C.POINTER(C.c_longlong), C.POINTER(C.c_longlong)]),
    "nib_net_set_tensor_core": (_i, [_vp, _i]),
    "nib_net_set_graph": (_i, [_vp, _i]),
    "nib_net_profile": (_i, [_vp, _i, _vp, _vp, _vp, _vp, _i, C.POINTER(_i), _vp]),
    "nib_score": (_i, [_vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
    "nib_score_table": (_i, [_vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "nib_tie_compact": (_i, [_vp, _i, C.c_float, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "nib_tie_scatter": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "nib_net_set_dynamic_batch": (_i, [_vp, _vp]),
    "nib_comm_unique_id": (_i, [_vp]),
    "nib_comm_init": (_i, [_vp, _i, _i, C.POINTER(_vp)]),
    "nib_comm_destroy": (_i, [_vp]),
    "nib_allgather_scores": (_i, [_vp, _vp, _i, _vp, _vp]),
    "nib_tc_gemm_bf16": (_i, [_vp, _vp, _vp, _i, _i, _i, _vp]),
    "nib_gp_gram_binary": (_i, [_vp, _i, _vp, _i, _i, _d, _d, _vp, _i, _vp]),
    "nib_gp_gram_rbf": (_i, [_vp, _i, _vp, _i, _i, _d, _d, _i, _vp, _i, _vp]),
    "nib_gp_cholesky": (_i, [_vp, _i, _i, _vp, _vp]),
    "nib_gp_trsm": (_i, [_vp, _i, _i, _vp, _i, _i, _i, _vp]),
    "nib_gp_dgemm_sub": (_i, [_vp, _vp, _vp, _i, _i, _i, _vp]),
    "nib_gp_posterior": (_i, [_vp, _i, _i, _vp, _vp, _i, _i, _d, _d, _d, _vp, _vp, _vp, _vp, _vp]),
    "nib_gp_lml": (_i, [_vp, _i, _i, _vp, _vp, C.POINTER(_d), _vp]),
    "nib_gp_lml_grad": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _d, C.POINTER(_d), _vp]),
    "nib_gp_lml_grad_rbf": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _d, C.POINTER(_d), _vp]),
    "nib_gp_ei": (_i, [_vp, _vp, _i, _d, _i, _vp, _vp, _vp]),
    "nib_gp_gemv_t": (_i, [_vp, _i, _i, _i, _vp, _vp, _vp]),
    "nib_gp_colsumsq": (_i, [_vp, _i, _i, _i, _vp, _vp]),
    "nib_gp_append_row": (_i, [_vp, _vp, _d, _vp, _vp, _i, _vp]),
    "nib_gp_kb_select": (_i, [_vp, _i, _vp, _i, _vp, _vp, _vp, _i, _i, _vp, _i, _i, _vp, _d, _d, _i, _d, _d, _vp, _vp,
                              _vp, _vp]),
    "nib_heatmap": (_i, [_vp, _i, _i, _i, _i, _vp, _i, _vp, _i, _vp, _vp]),
    "nib_heatmap_pixels": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp]),
    "nib_ski_accumulate": (_i, [_vp, _vp, _i, _d, _d, _i, _d, _vp, _vp, _vp]),
    "nib_ski_predict": (_i, [_vp, _i, _d, _d, _i, _d, _vp, _vp, _d, _i, _vp, _vp, _vp]),
    "nib_ski_kron_apply": (_i, [_vp, _vp, _i, _i, _vp, _vp, _i, _vp, _vp]),
    "nib_ski_band_accumulate": (_i, [_vp, _vp, _i, _d, _d, _i, _d, _vp, _vp, _vp, _vp]),
    "nib_ski_band_spmv": (_i, [_vp, _i, _vp, _vp, _i, _vp]),
    "nib_ski_kron_pcg": (_i, [_vp, _i, _vp, _vp, _vp, _vp, _d, _d, _vp, _vp, _i, _d, _i, _i, _vp, C.POINTER(_i),
                              C.POINTER(_d), _vp]),
    "nib_ski_kron_var_rhs": (_i, [_vp, _i, _d, _d, _i, _vp, _vp, _vp, _vp]),
    "nib_ski_kron_var_reduce": (_i, [_vp, _vp, _i, _i, _d, _i, _vp, _vp]),
    "nib_segment_weights": (_i, [_vp, _i, _vp, _i, _i, _vp, _vp, _vp]),
    "nib_heat_normalize_u8": (_i, [_vp, _i, _vp, _vp, _vp]),
    "nib_threshold_bbox": (_i, [_vp, _i, _i, _i, _vp, _vp]),
    "nib_vgp_loglik_grad": (_i, [_vp, _vp, _i, _d, _d, _i, _d, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "nib_vgp_predict": (_i, [_vp, _i, _d, _d, _i, _d, _vp, _vp, _vp, _vp, _vp, _vp]),
    "nib_felzenszwalb": (_i, [_vp, _i, _i, _i, _d, _d, _i, _vp, C.POINTER(_i)]),
}

EXPORTED_SYMBOLS = tuple(_PROTOTYPES)

_lib = None


def load() -> C.CDLL:
    """Load libnib.so, raising loudly if it has not been built (python -m ...build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -m network_interpretation_imagenet_b200.build` "
            "(nvcc, sm_100a).  There is no CPU/PyTorch fallback for this engine.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in _PROTOTYPES.items():
        fn = getattr(lib, name)  # AttributeError if the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    if lib.nib_abi_version() != ABI_VERSION:
        raise ImportError(f"libnib.so ABI version {lib.nib_abi_version()} != {ABI_VERSION}; rebuild")
    _lib = lib
    return lib


def check(code: int, where: str) -> None:
    if code != NIB_OK:
        msg = load().nib_last_error()
        raise NibError(code, where, msg.decode("utf-8", "replace") if msg else "")


def ptr(t) -> int | None:
    """Device (or host) address of a torch tensor / numpy array, None passthrough."""
    if t is None:
        return None
    if hasattr(t, "data_ptr"):
        return t.data_ptr()
    return t.ctypes.data


def stream_handle(stream=None) -> int:
    import torch

    s = stream if stream is not None else torch.cuda.current_stream()
    return s.cuda_stream
