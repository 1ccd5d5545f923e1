"""ctypes binding of the C ABI declared in include/lzb200.h (liblzb200.so).

There is NO fallback: if the CUDA library is missing or no device is present, importing callers get
a loud RuntimeError -- the product path never routes through PyTorch eager or the CPU oracle.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# LZ_LIB_TAG=NAME selects an experiment build (_lib/NAME/liblzb200.so, see _build.py); still the CUDA library, never a fallback
LIB_PATH = os.path.join(_HERE, "_lib", os.environ.get("LZ_LIB_TAG", ""), "liblzb200.so")
_lib = None

c_int, c_float, c_void_p, c_char_p, c_int64 = (ctypes.c_int, ctypes.c_float, ctypes.c_void_p,
                                               ctypes.c_char_p, ctypes.c_int64)


class ModelConfig(ctypes.Structure):
    """struct lz_model_config (include/lzb200.h)"""
    _fields_ = [("obs_c", c_int), ("obs_h", c_int), ("obs_w", c_int), ("action_space_size", c_int),
                ("num_res_blocks", c_int), ("num_channels", c_int), ("reward_head_channels", c_int),
                ("value_head_channels", c_int), ("policy_head_channels", c_int), ("reward_hidden", c_int),
                ("value_hidden", c_int), ("policy_hidden", c_int), ("support_min", c_float),
                ("support_max", c_float), ("support_step", c_float), ("efficientzero", c_int), ("lstm_hidden_size", c_int)]


class MlpConfig(ctypes.Structure):
    """struct lz_mlp_config (include/lzb200.h)"""
    _fields_ = [("obs_dim", c_int), ("action_space_size", c_int), ("latent_dim", c_int), ("reward_hidden", c_int),
                ("value_hidden", c_int), ("policy_hidden", c_int), ("res_connection_in_dynamics", c_int),
                ("support_min", c_float), ("support_max", c_float), ("support_step", c_float)]


# name -> (restype, argtypes); every symbol include/lzb200.h declares
SIGNATURES = {
    "lz_version": (c_int, []),
    "lz_debug_launch_count": (ctypes.c_uint64, []),
    "lz_last_error": (c_char_p, []),
    "lz_tree_create": (c_int, [c_int, c_int, c_int, ctypes.POINTER(c_void_p)]),
    "lz_tree_destroy": (c_int, [c_void_p]),
    "lz_tree_set_params": (c_int, [c_void_p, c_int, c_float, c_float, c_float]),
    "lz_tree_reset": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p]),
    "lz_tree_reset_mask": (c_int, [c_void_p, c_void_p, c_void_p]),
    "lz_tree_prepare": (c_int, [c_void_p, c_void_p, c_void_p, c_float, c_void_p, c_void_p, c_void_p]),
    "lz_tree_traverse": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "lz_tree_backpropagate": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "lz_tree_traverse_with_reuse": (c_int, [c_void_p] * 9),
    "lz_tree_backpropagate_with_reuse": (c_int, [c_void_p, c_int] + [c_void_p] * 8),
    "lz_tree_select_action": (c_int, [c_void_p, c_float, c_int, ctypes.c_uint64, c_void_p, c_void_p, c_void_p, c_void_p]),
    "lz_tree_set_ez": (c_int, [c_void_p, c_int, c_int]),
    "lz_tree_set_tiebreak": (c_int, [c_void_p, c_int]),
    "lz_tree_traverse_ez": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "lz_tree_backpropagate_ez": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "lz_tree_results": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "lz_tree_set_gumbel": (c_int, [c_void_p, c_int, c_int]),
    "lz_tree_prepare_gumbel": (c_int, [c_void_p, c_void_p, c_void_p, c_float, c_void_p, c_void_p, c_void_p, c_void_p]),
    "lz_tree_traverse_gumbel": (c_int, [c_void_p, c_float, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "lz_tree_backpropagate_gumbel": (c_int, [c_void_p, c_int, c_float, c_void_p, c_void_p, c_void_p, c_void_p]),
    "lz_tree_results_gumbel": (c_int, [c_void_p, c_float, c_void_p, c_void_p, c_void_p, c_void_p]),
    "lz_model_create": (c_int, [ctypes.POINTER(ModelConfig), ctypes.POINTER(c_void_p)]),
    "lz_model_create_mlp": (c_int, [ctypes.POINTER(MlpConfig), ctypes.POINTER(c_void_p)]),
    "lz_model_destroy": (c_int, [c_void_p]),
    "lz_model_set_tensor": (c_int, [c_void_p, c_char_p, c_void_p, c_int64]),
    "lz_model_finalize": (c_int, [c_void_p]),
    "lz_model_set_math": (c_int, [c_void_p, c_int]),
    "lz_model_debug_tc_program": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p, c_int]),
    "lz_debug_tc_stamps": (c_int, [c_void_p]),
    "lz_model_latent_hw": (c_int, [c_void_p]),
    "lz_model_support_size": (c_int, [c_void_p]),
    "lz_model_initial_inference": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "lz_model_recurrent_inference": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                             c_void_p, c_void_p, c_void_p, c_void_p]),
    "lz_model_recurrent_inference_ez": (c_int, [c_void_p, c_int] + [c_void_p] * 12 + [c_void_p]),
    "lz_model_lstm_hidden_size": (c_int, [c_void_p]),
    "lz_inverse_scalar_transform": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p]),
    "lz_search_create": (c_int, [c_void_p, c_void_p, c_int, ctypes.POINTER(c_void_p)]),
    "lz_search_destroy": (c_int, [c_void_p]),
    "lz_search_run": (c_int, [c_void_p, c_void_p, c_int, c_void_p]),
    "lz_search_collect": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_float, c_void_p, c_int, c_void_p,
                                  c_void_p, c_void_p]),
    "lz_search_collect_host": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_float, c_void_p, c_int, c_int, c_void_p,
                                       c_void_p, c_void_p]),
    "lz_search_collect_u8": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_float, c_void_p, c_int, c_void_p,
                                     c_void_p, c_void_p]),
    "lz_search_collect_host_u8": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_float, c_void_p, c_int, c_int, c_void_p,
                                          c_void_p, c_void_p]),
    "lz_search_num_kernels": (c_int, [c_void_p]),
    "lz_search_latent_pool": (c_void_p, [c_void_p]),
    "lz_search_run_with_reuse": (c_int, [c_void_p] * 6),
    "lz_search_run_gumbel": (c_int, [c_void_p, c_void_p, c_float, c_void_p]),
    "lz_search_run_ez": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "lz_search_run_ez_with_reuse": (c_int, [c_void_p] * 8),
    "lz_frames_create": (c_int, [c_int, c_int, c_int, c_int, ctypes.POINTER(c_void_p)]),
    "lz_frames_destroy": (c_int, [c_void_p]),
    "lz_frames_push": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p]),
    "lz_frames_push_host": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p]),
    "lz_frames_stacked": (c_void_p, [c_void_p]),
    "lz_segments_create": (c_int, [c_int, c_int, c_int, ctypes.POINTER(c_void_p)]),
    "lz_segments_destroy": (c_int, [c_void_p]),
    "lz_segments_store_search_stats": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "lz_segments_reset": (c_int, [c_void_p, c_void_p, c_void_p]),
    "lz_segments_data": (c_int, [c_void_p, ctypes.POINTER(c_void_p), ctypes.POINTER(c_void_p), ctypes.POINTER(c_void_p)]),
    "lz_search_hidden_pool": (c_void_p, [c_void_p, c_int]),
}


def load():
    """Loads liblzb200.so and types every entry point.  Raises if the library was not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  lightzero_b200 has no CPU / PyTorch fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)   # AttributeError here == header / library mismatch
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


class LzError(RuntimeError):
    pass


def check(rc: int, what: str = ""):
    if rc < 0:
        msg = load().lz_last_error()
        raise LzError(f"{what} failed ({rc}): {msg.decode() if msg else ''}")
    return rc


def ptr(t):
    """Device/host pointer of a tensor (or None)."""
    return None if t is None else t.data_ptr()


def stream_ptr():
    import torch
    return torch.cuda.current_stream().cuda_stream
