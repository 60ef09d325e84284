"""ctypes binding of libsniper_b200.so (the C-ABI declared in include/sniper_b200.h).

The product path has no CPU fallback: if the library is missing, loading raises.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libsniper_b200.so")

_T = {"p": ctypes.c_void_p, "i": ctypes.c_int, "l": ctypes.c_long, "f": ctypes.c_float, "z": ctypes.c_size_t,
      "d": ctypes.c_double, "u": ctypes.c_uint}

# name -> (restype code, argument codes); order and meaning documented in include/sniper_b200.h
SIGNATURES = {
    "sniper_last_error": ("s", ""),
    "sniper_abi_version": ("i", ""),
    "sniper_multi_proposal_target_workspace_bytes": ("z", "iiii"),
    "sniper_generate_anchors": ("i", "ipipip"),
    "sniper_proposal_decode": ("i", "pppp" "iiiii" "pipi" "iii" "ppp" "p"),
    "sniper_multi_proposal_target_fwd": ("i", "ppppp" "iiiiiii" "pipi" "f" "iii" "pppp" "pp" "pz" "p"),
    "sniper_multi_proposal_workspace_bytes": ("z", "iiiii"),
    "sniper_multi_proposal_fwd": ("i", "ppp" "iiiiiii" "pipi" "f" "i" "f" "iii" "pppp" "pz" "p"),
    "sniper_deform_psroi_fwd": ("i", "ppp" "iiii" "f" "iiiii" "f" "iii" "ppp" "p"),
    "sniper_deform_psroi_bwd": ("i", "pppp" "iiii" "f" "iiiii" "f" "iii" "pp" "p"),
    "sniper_deform_psroi_fwd_tiled": ("i", "ppp" "iiiii" "f" "iiiii" "f" "ii" "pp" "p"),
    "sniper_deform_psroi_bwd_tiled_workspace_bytes": ("z", "iiii"),
    "sniper_deform_psroi_bwd_tiled": ("i", "pppp" "iiiii" "f" "iiiii" "f" "ii" "pp" "pz" "p"),
    "sniper_psroi_fwd": ("i", "pp" "iiii" "f" "iiii" "pp" "p"),
    "sniper_psroi_bwd": ("i", "pp" "iiii" "f" "iiii" "p" "p"),
    "sniper_gemm_nt": ("i", "plplpl" "iiii" "ppp" "l" "iii" "pp"),
    "sniper_gemm_plan": ("i", "iiiip"),
    "sniper_gemm_tail_workspace_bytes": ("z", ""),
    "sniper_gemm_set_tail_workspace": ("i", "pzi"),
    "sniper_conv2d_nhwc": ("i", "pliiii" "pii" "pp" "iii" "pl" "iiiii" "i" "ppp" "l" "iii" "pp"),
    "sniper_conv2d_wgrad_nhwc": ("i", "plpl" "iiiii" "i" "pp" "iii" "p" "ii" "p"),
    "sniper_affine_act": ("i", "plpppl" "l" "iii" "p"),
    "sniper_bn_stats": ("i", "pllippffipppppppip"),
    "sniper_bn_finalize": ("i", "plippffippppppp"),
    "sniper_bn_apply_train": ("i", "plplippffippppppplii" "p"),
    "sniper_bn_frozen": ("i", "ippppfippp"),
    "sniper_bn_relu_bwd": ("i", "plplppppp" "pl" "pl" "pp" "lii" "p"),
    "sniper_bn_act_bwd": ("i", "plplppppp" "pl" "pl" "pp" "liii" "p"),
    "sniper_affine_relu_bwd": ("i", "plplpp" "pl" "pl" "lii" "p"),
    "sniper_depthwise3x3_fwd": ("i", "plppl" "iiiiii" "p"),
    "sniper_depthwise3x3_dgrad": ("i", "plppl" "iiiiii" "p"),
    "sniper_depthwise3x3_wgrad": ("i", "plplp" "iiiiii" "p"),
    "sniper_im2col3x3s2_nchw": ("i", "pp" "iiiiii" "p"),
    "sniper_add_rows": ("i", "plplpl" "lii" "p"),
    "sniper_relu_bwd": ("i", "plplplli" "i" "p"),
    "sniper_cast_rows": ("i", "plipli" "li" "p"),
    "sniper_maxpool3x3s2_nhwc": ("i", "ppiiiiip"),
    "sniper_stem_conv": ("i", "pppppppiiiip"),
    "sniper_stem_im2col": ("i", "pppp" "iiiii" "p"),
    "sniper_weight_transpose": ("i", "ppiiiipp"),
    "sniper_weight_transpose_batched": ("i", "piip"),
    "sniper_bn_param_grad_batched": ("i", "pip"),
    "sniper_colsum": ("i", "pllipp"),
    "sniper_sgd_mom": ("i", "ppplffffp"),
    "sniper_sgd_mom_dev": ("i", "ppplpffffpp"),
    "sniper_count_valid": ("i", "plipp"),
    "sniper_rpn_softmax_loss": ("i", "pipiiiifppipipp"),
    "sniper_rpn_smooth_l1_loss": ("i", "pippiiiifpipp"),
    "sniper_softmax_ce": ("i", "pipiiifppipipp"),
    "sniper_smooth_l1_loss": ("i", "pipplifpipp"),
    "sniper_focus_head": ("i", "pli" "ppp" "f" "p" "pppp" "p" "p"),
    "sniper_deform_im2col": ("i", "pp" "iiiiiiiiiii" "pip"),
    "sniper_deform_col2im": ("i", "ppp" "iiiiiiiiiii" "ppip"),
    "sniper_anchor_target": ("i", "ppippipp" "iiii" "pipi" "dd" "ppppp" "p"),
    "sniper_soft_nms_batched": ("i", "ppifffuppp"),
    "sniper_chip_input": ("i", "ppppiip"),
    "sniper_chip_input_hw": ("i", "ppppiiip"),
    "sniper_anchor_subsample": ("i", "pppiiiiiiup"),
    "sniper_focus_label": ("i", "pp" "iiii" "ddd" "p" "p"),
    "sniper_chips_generate": ("i", "piiiiipi"),
    "sniper_cpu_nms": ("i", "ppidp"),
    "sniper_cpu_soft_nms": ("i", "pifffu"),
    "sniper_bbox_overlaps": ("i", "pipipi"),
}

_lib = None

# GPU kernels launched per C-ABI call (host-only entry points: 0)
KERNELS_PER_CALL = {
    "sniper_last_error": 0, "sniper_abi_version": 0, "sniper_multi_proposal_target_workspace_bytes": 0,
    "sniper_generate_anchors": 0, "sniper_chips_generate": 0, "sniper_cpu_nms": 0, "sniper_cpu_soft_nms": 0,
    "sniper_bbox_overlaps": 0, "sniper_gemm_plan": 0, "sniper_deform_psroi_bwd_tiled_workspace_bytes": 0, "sniper_gemm_tail_workspace_bytes": 0, "sniper_gemm_set_tail_workspace": 0, "sniper_multi_proposal_target_fwd": 2, "sniper_multi_proposal_workspace_bytes": 0, "sniper_multi_proposal_fwd": 4, "sniper_anchor_target": 2, "sniper_bn_stats": 2, "sniper_bn_relu_bwd": 2, "sniper_bn_act_bwd": 2,
}
launches = [0]


class _Counting(object):
    """Thin proxy over the CDLL that counts the GPU kernels our entry points launch (bench.py gpu_launches)."""

    def __init__(self, cdll):
        self._cdll = cdll
        self._cache = {}

    def __getattr__(self, name):
        fn = self._cache.get(name)
        if fn is None:
            raw = getattr(self._cdll, name)
            k = KERNELS_PER_CALL.get(name, 1)

            def fn(*a, _raw=raw, _k=k):
                launches[0] += _k
                return _raw(*a)
            self._cache[name] = fn
        return fn


def lib():
    """Returns the loaded C-ABI library; raises (loudly) if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "sniper_b200: %s is missing -- run `python -m sniper_b200.build` (there is no CPU fallback)" % LIB_PATH)
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = ctypes.c_char_p if res == "s" else _T[res]
            fn.argtypes = [_T[c] for c in args]
        _lib = _Counting(L)
    return _lib


class SniperError(RuntimeError):
    """Raised when a C-ABI entry point returns non-zero (MXNetError analogue)."""


def check(rc):
    if rc != 0:
        raise SniperError(lib().sniper_last_error().decode())
