"""ctypes binding of libcvcl_b200.so (the C ABI declared in include/cvcl_b200.h).

There is no CPU implementation behind these functions: if the shared library is missing the
import of the ops fails loudly (`CvclLibraryMissing`), and every call requires CUDA tensors.
"""
import ctypes
import os
from ctypes import c_float, c_int, c_int64, c_size_t, c_void_p, c_char_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libcvcl_b200.so")
ABI_VERSION = 6


class CvclLibraryMissing(RuntimeError):
    pass


class CvclError(RuntimeError):
    pass


_P = c_void_p
_I = c_int
_F = c_float
_L = c_int64

# name -> (restype, argtypes); must list every symbol include/cvcl_b200.h declares
PROTOTYPES = {
    "cvcl_abi_version": (c_int, []),
    "cvcl_last_error": (c_char_p, []),
    "cvcl_launch_count": (ctypes.c_ulonglong, []),
    "cvcl_host_alloc": (c_void_p, [c_size_t, _I]),
    "cvcl_host_free": (c_int, [_P]),
    "cvcl_text_encoder_fwd": (c_int, [_P, _P, _P, _I, _I, _I, _I, _I, _I, _F, _P, _P, _I, _P,
                                      _P, _P, _P, _P]),
    "cvcl_embedding_gather": (c_int, [_P, _P, _P, _I, _I, _I, _P]),
    "cvcl_embedding_scatter_add": (c_int, [_P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "cvcl_embedding_bag_bwd": (c_int, [_P, _P, _P, _P, _P, _I, _P, _I, _I, _I, _I, _P]),
    "cvcl_text_token_bwd": (c_int, [_P, _P, _P, _P, _P, _F, _P, _I, _I, _I, _I, _I, _P]),
    "cvcl_cast_transpose": (c_int, [_P, _I, _P, _P, _I, _I, _I, _L, _L, _L, _L, _L, _L, _P]),
    "cvcl_rownorm_bwd": (c_int, [_P, _P, _P, _I, _I, _I, _P, _P, _I, _P, _I, _P, _P]),
    "cvcl_spatial_pool": (c_int, [_P, _I, _I, _I, _P, _P, _I, _P, _I, _P]),
    "cvcl_spatial_pool_bwd": (c_int, [_P, _I, _I, _I, _P, _P]),
    "cvcl_linear_f32": (c_int, [_P, _I, _P, _I, _P, _I, _I, _I, _P, _I, _P]),
    "cvcl_normalize_rows_f32": (c_int, [_P, _P, _L, _I, _P]),
    "cvcl_row_argmax_f32": (c_int, [_P, _L, _L, _I, _I, _I, _P, _P, _P]),
    "cvcl_rank_topk_f32": (c_int, [_P, _L, _L, _I, _L, _P, _P, _I, _P, _P, _P, _P]),
    "cvcl_head_proj_norm_fwd": (c_int, [_P, _I, _P, _I, _P, _I, _I, _I, _I, _P, _I, _P, _I, _P, _P]),
    "cvcl_sim_workspace_bytes": (c_size_t, [_I, _I, _I, _I]),
    "cvcl_sim_infonce_fwd": (c_int, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _F, _I, _F, _P, _P, _P, _P,
                                     _P, _P, _I, _P]),
    "cvcl_sim_logits_fwd": (c_int, [_P, _P, _I, _I, _I, _I, _F, _P, _P, _P]),
    "cvcl_sim_infonce_bwd_g": (c_int, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _F, _I, _F, _P, _P, _P, _P,
                                       _P, _I, _P, _I, _P, _P, _P, _P]),
    "cvcl_feat_grad_norm_bwd": (c_int, [_P, _I, _I, _P, _I, _I, _I, _I, _P, _I, _P, _I, _P, _P, _I, _I, _I,
                                        _P, _P, _I, _P, _I, _P, _P]),
    "cvcl_feat_grad_norm_bwd_ws": (c_int, [_P, _I, _I, _P, _I, _I, _I, _I, _P, _I, _P, _I, _P, _P, _I, _I, _I,
                                           _P, _P, _I, _P, _I, _P, _P, _P]),
    "cvcl_head_weight_grad": (c_int, [_P, _I, _P, _I, _I, _I, _I, _P, _I, _P]),
    "cvcl_gemm_f32out": (c_int, [_P, _I, _I, _P, _I, _I, _I, _I, _I, _F, _P, _I, _P]),
    "cvcl_flat_step_workspace_bytes": (c_size_t, [_I, _I, _I, _I, _I]),
    "cvcl_flat_step_layout": (c_int, [_I, _I, _I, _I, _I, _P, _I]),
    "cvcl_flat_contrastive_step": (c_int, [_P, _I, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _F, _I, _P,
                                           _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "cvcl_flat_fused_supported": (c_int, [_I, _I, _I, _I, _I]),
    "cvcl_flat_fused_workspace_bytes": (c_size_t, [_I, _I, _I, _I, _I]),
    "cvcl_flat_fused_layout": (c_int, [_I, _I, _I, _I, _I, _P, _I]),
    "cvcl_flat_step_fused": (c_int, [_P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _F, _P, _I, _P, _P, _P,
                                     _P, _P, _P, _P, _P, _P, _I, _P]),
    "cvcl_flat_fused_sharded_supported": (c_int, [_I, _I, _I, _I, _I, _I]),
    "cvcl_flat_fused_sharded_workspace_bytes": (c_size_t, [_I, _I, _I, _I, _I, _I]),
    "cvcl_flat_fused_sharded_part_bytes": (c_size_t, [_I, _I]),
    "cvcl_flat_fused_sharded_scratch_bytes": (c_size_t, [_I, _I, _I, _I, _I, _I]),
    "cvcl_flat_step_fused_sharded": (c_int, [_P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _F, _P, _I, _P, _P, _P,
                                             _P, _P, _P, _P, _P, _P, _I, _I, _I, _P, _P, _P, _P, _P, _P, _P,
                                             _L, _P]),
    "cvcl_spatial_max_fwd": (c_int, [_P, _P, _P, _I, _I, _I, _I, _I, _P, _P, _P, _P]),
    "cvcl_spatial_max_bwd_workspace_bytes": (c_size_t, [_I, _I, _I, _I, _I]),
    "cvcl_spatial_max_bwd": (c_int, [_P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P, _P, _P, _P]),
    "cvcl_match_infonce_fwd": (c_int, [_P, _I, _F, _F, _P, _P, _P, _P, _P, _P, _P]),
    "cvcl_match_infonce_bwd": (c_int, [_P, _I, _F, _F, _P, _P, _P, _P, _P]),
    "cvcl_match_infonce_block_fwd": (c_int, [_P, _P, _I, _I, _I, _F, _F, _P, _P, _P, _P, _P, _P, _P]),
    "cvcl_match_infonce_block_bwd_workspace_bytes": (c_size_t, [_I, _I]),
    "cvcl_match_infonce_block_bwd": (c_int, [_P, _P, _I, _I, _I, _F, _F, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "cvcl_p2p_gather": (c_int, [_P, _I, _I, ctypes.c_longlong, _P, ctypes.c_longlong, _P]),
    "cvcl_peer_flag_words": (c_size_t, []),
    "cvcl_peer_max_blocks": (c_int, []),
    "cvcl_peer_allgather": (c_int, [_P, _P, _P, _P, _I, _I, ctypes.c_longlong, _I, ctypes.c_longlong, _P,
                                    ctypes.c_longlong, ctypes.c_uint, _P]),
    "cvcl_peer_allreduce_f32": (c_int, [_P, _P, _P, _P, _I, _I, ctypes.c_longlong, ctypes.c_uint, _P]),
    "cvcl_peer_allgather_push": (c_int, [_P, _P, _P, _P, _I, _I, _P, ctypes.c_longlong, _I, ctypes.c_longlong,
                                         ctypes.c_longlong, ctypes.c_uint, _P]),
    "cvcl_peer_allreduce_scratch_bytes": (c_size_t, [ctypes.c_longlong, _I]),
    "cvcl_peer_allreduce_push_f32": (c_int, [_P, _P, _P, _P, _P, _I, _I, ctypes.c_longlong, ctypes.c_uint, _P]),
    "cvcl_peer_barrier": (c_int, [_P, _P, _P, _I, _I, ctypes.c_uint, _P]),
    "cvcl_adamw_step": (c_int, [_P, _P, _P, _P, ctypes.c_longlong, _F, _F, _F, _F, _F, _I, _F, _P, _P]),
    "cvcl_adamw_multi_step": (c_int, [_I, _P, _P, _P, _P, _P, _P, _P, _P, _F, _F, _F, _F, _P, _P, _P]),
    "cvcl_gradcam_workspace_bytes": (c_size_t, [_I, _I, _I]),
    "cvcl_gradcam_flat": (c_int, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _P, _P, _P]),
    "cvcl_bicubic_upsample": (c_int, [_P, _I, _I, _I, _I, _I, _P, _P]),
    "cvcl_eval_nway_fwd": (c_int, [_P, _P, _P, _I, _I, _I, _I, _F, _P, _P, _P]),
    "cvcl_conv1x1_f32": (c_int, [_P, _P, _P, _I, _I, _I, _I, _P, _P]),
    "cvcl_spatial_max_scores_f32": (c_int, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _F, _P, _P]),
    "cvcl_spatial_attention_f32": (c_int, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _P, _P, _P, _P]),
}

_lib = None


def load(path=None):
    """dlopen the library and attach prototypes; raises CvclLibraryMissing if absent."""
    global _lib
    if _lib is not None:
        return _lib
    explicit = path or os.environ.get("CVCL_B200_LIB")
    path = explicit or LIB_PATH
    if not explicit:
        # in-tree build on first use, and again when a source is newer than the library (nvcc
        # cross-compiles sm_100a anywhere; locked + atomic rename, see build.py); still no CPU path
        try:
            from . import build as _build
            if _build.is_stale():
                _build.build_library()
        except Exception as exc:                                   # noqa: BLE001
            if not os.path.exists(path):
                raise CvclLibraryMissing("libcvcl_b200.so is missing and could not be built: %s" % exc)
    if not os.path.exists(path):
        raise CvclLibraryMissing(
            "libcvcl_b200.so not found at %s -- build it with `python multimodal-baby_b200/build.py` "
            "(there is no CPU fallback for the cvcl_b200 ops)" % path)
    lib = ctypes.CDLL(path)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)          # AttributeError if the header and the .so disagree
        fn.restype = res
        fn.argtypes = args
    v = lib.cvcl_abi_version()
    if v != ABI_VERSION:
        raise CvclError("libcvcl_b200 ABI version %d, bindings expect %d" % (v, ABI_VERSION))
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        msg = load().cvcl_last_error()
        raise CvclError("libcvcl_b200 error %d: %s" % (rc, (msg or b"").decode(errors="replace")))


def call(name, *args):
    check(getattr(load(), name)(*args))
