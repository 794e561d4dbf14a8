"""ctypes binding of ``libosb200.so`` (the C ABI declared in ``include/osb200.h``).

The library is the product: there is no Python/torch fallback.  If the shared object is missing
or a call fails, a RuntimeError is raised with the library's own error string.
"""
import ctypes
import os
from ctypes import c_char_p, c_double, c_int, c_int32, c_int64, c_size_t, c_void_p, POINTER

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libosb200.so')
_lib = None

P = c_void_p     # noqa: E305 (re-exported as _cabi.c_void_p)
I32, I64, SZ = c_int32, c_int64, c_size_t

# name -> (restype, argtypes); mirrors include/osb200.h one to one
SIGNATURES = {
    'osb_version': (c_int, []),
    'osb_last_error': (c_char_p, []),
    'osb_device_info': (c_int, [POINTER(c_int), POINTER(c_int), POINTER(c_int)]),
    'osb_launch_count': (I64, []),
    'osb_measure_sm_mhz': (c_int, [P, P]),
    'osb_coordset_workspace_bytes': (SZ, [I64]),
    'osb_coordset_build': (c_int, [P, I64, P, P, P, P, I64, POINTER(I32), P, SZ, P]),
    'osb_coordset_stride': (c_int, [P, I64, I32, P, P, POINTER(I64), P, SZ, P]),
    'osb_coordset_pyramid': (c_int, [P, I64, I32, P, P, P, P, I64, P, P, POINTER(I64), POINTER(I32), P, SZ, P]),
    'osb_hash_build': (c_int, [P, I64, P, I64, P]),
    'osb_kernel_map_build': (c_int, [P, I64, P, I64, I32, I32, I32, I32, P, P, P]),
    'osb_kernel_map_transpose': (c_int, [P, I64, I32, P, I64, P]),
    'osb_conv_fwd_f32': (c_int, [P, I64, P, I64, I32, P, I32, I32, I32, P, P]),
    'osb_conv_wgrad_f32': (c_int, [P, P, I64, I32, P, I32, I32, P, P]),
    'osb_conv_wgrad_tc_workspace_bytes': (SZ, [I64, I32, I32, I32]),
    'osb_conv_wgrad_tc': (c_int, [P, I32, I64, P, I64, I32, P, I32, P, P, SZ, P]),
    'osb_conv_packed_weight_bytes': (SZ, [I32, I32, I32]),
    'osb_conv_pack_weights': (c_int, [P, I32, I32, I32, I32, P, P]),
    'osb_conv_tc_workspace_bytes': (SZ, [I64, I32, I32, I32]),
    'osb_conv_fwd_tc': (c_int, [P, I32, I64, P, I32, I64, P, I64, I32, P, I32, P, P, P, I32, P, P, P, P, SZ, I32, P]),
    'osb_convtr_fwd_tc': (c_int, [P, I32, I64, P, I32, P, I32, P, P, I32, P, P, I32, P]),
    'osb_conv_desc_bytes': (SZ, []),
    'osb_conv_weight_tiles_bytes': (SZ, [I32, I32, I32]),
    'osb_conv_pack_weight_tiles': (c_int, [P, I32, I32, I32, I32, P, P]),
    'osb_conv_chain_grid': (c_int, []),
    'osb_conv_chain_workspace_bytes': (SZ, [I64, I32, I32, I32]),
    'osb_conv_desc_fill': (c_int, [P, P, I32, P, I32, P, I64, I32, P, I32, P, P, P, I32, P, P, P, P, I32, P, SZ, I32]),
    'osb_conv_chain_launch': (c_int, [P, I32, P, I32, P]),
    'osb_tuning_set': (c_int, [c_char_p, I64]),
    'osb_conv_stem_fused': (c_int, [P, I32, P, I64, P, I64, I32, I32, P, I32, P, P, I32, P, P, P]),
    'osb_f32_to_split': (c_int, [P, I64, I32, P, P]),
    'osb_split_to_f32': (c_int, [P, I64, I32, P, P]),
    'osb_gather_rows_f32': (c_int, [P, P, I64, I32, P, P]),
    'osb_match_scores': (c_int, [P, I32, I64, I32, P, I64, P, I32, I32, P, P, P, P]),
    'osb_match_ensemble': (c_int, [P, P, I64, I32, P, I64, P, P, P, I32, P, P, P, P]),
    'osb_match_accumulate': (c_int, [P, I32, P, P, P, I64, I32, P, I64, P, I32, I32, P, I32, P, P]),
    'osb_logits_accumulate': (c_int, [P, I64, I32, P, I64, P, I32, P, P, P]),
    'osb_folded_head_finish': (c_int, [P, I64, I32, I32, I32, P, P, P, P]),
    'osb_voxelize_workspace_bytes': (SZ, [I64]),
    'osb_voxelize': (c_int, [P, I32, I64, POINTER(c_double), P, P, P, POINTER(I64), POINTER(c_double), P, SZ, P]),
    'osb_occgrid_bytes': (SZ, [I32, I32]),
    'osb_occgrid_build': (c_int, [P, I64, I32, I32, I32, P, P, P]),
    'osb_kernel_map_build_grid': (c_int, [P, I64, P, I32, I32, I32, I32, I32, I32, I32, P, P, P]),
    'osb_conv_stem_fused_grid': (c_int, [P, I32, P, I64, P, I32, I32, I32, I32, I32, P, I32, P, P, I32, P, P, P]),
    'osb_fusion_workspace_bytes': (SZ, [I64, I32]),
    'osb_fusion_accumulate': (c_int, [P, I32, I64, P, P, P, P, I32, I32, I32, I32, I32, c_double, P, P, P, P, SZ, P]),
    'osb_fusion_finalize': (c_int, [P, P, I64, I32, P, P]),
    'osb_feature_remap_workspace_bytes': (SZ, [I64, I64]),
    'osb_feature_remap': (c_int, [P, I64, P, I64, P, I64, I32, I32, P, P, POINTER(I64), P, SZ, P]),
    'osb_confusion_accumulate': (c_int, [P, P, I32, I64, I32, I32, I32, P, P, P]),
    'osb_intersection_union': (c_int, [P, P, I32, I64, I32, I32, P, P]),
}


def lib():
    """Load libosb200.so once; raise loudly when it is missing (no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"openscene_b200: native library {LIB_PATH} is missing. Build it with "
                f"`python -c 'import __graft_entry__ as g; g.build()'` (nvcc, sm_100a). "
                f"There is no CPU/PyTorch fallback for this path.")
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)          # AttributeError here = header/library mismatch
            fn.restype, fn.argtypes = res, args
        _lib = L
    return _lib


def check(rc, what):
    if rc != 0:
        msg = lib().osb_last_error()
        raise RuntimeError(f"{what} failed: {msg.decode() if msg else 'unknown error'}")


def call(name, *args):
    check(getattr(lib(), name)(*args), name)


def ptr(t):
    """Raw device pointer of a torch tensor (None -> NULL)."""
    if t is None:
        return None
    return c_void_p(t.data_ptr())


def stream_ptr():
    import torch
    return c_void_p(torch.cuda.current_stream().cuda_stream)


def require_cuda(t, what):
    if not t.is_cuda:
        raise RuntimeError(f"openscene_b200: {what} must be a CUDA tensor (got device {t.device}); "
                           f"there is no CPU fallback for this path")
