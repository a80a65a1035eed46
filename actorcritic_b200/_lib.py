"""ctypes binding of libacx.so (the C ABI in include/acx.h).

The library is the product: if it is missing or does not load, importing anything that computes
raises - there is no CPU or PyTorch fallback.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libacx.so")

MAX_PLANES = 3


class AcxError(RuntimeError):
    pass


class Planes(ctypes.Structure):
    _fields_ = [("planes", ctypes.c_void_p * MAX_PLANES), ("num_planes", ctypes.c_int),
                ("rows", ctypes.c_int), ("cols", ctypes.c_int), ("ld", ctypes.c_int)]


class Gather(ctypes.Structure):
    _fields_ = [("planes", ctypes.c_void_p * MAX_PLANES), ("num_planes", ctypes.c_int),
                ("dim", ctypes.c_longlong * 5), ("stride_bytes", ctypes.c_longlong * 4),
                ("gx", ctypes.c_int), ("gy", ctypes.c_int), ("samples", ctypes.c_int), ("num_chunks", ctypes.c_int),
                ("c0", ctypes.c_byte * 16), ("c1", ctypes.c_byte * 16), ("c2", ctypes.c_byte * 16), ("c3", ctypes.c_byte * 16)]


class Gemm(ctypes.Structure):
    _fields_ = [("a", Planes), ("b", Planes), ("trans_a", ctypes.c_int), ("trans_b", ctypes.c_int),
                ("m", ctypes.c_int), ("n", ctypes.c_int), ("k", ctypes.c_int),
                ("num_pairs", ctypes.c_int), ("pair_a", ctypes.c_int * 6), ("pair_b", ctypes.c_int * 6),
                ("alpha", ctypes.c_float), ("bias", ctypes.c_void_p), ("relu", ctypes.c_int),
                ("symmetric", ctypes.c_int),
                ("c", ctypes.c_void_p), ("ldc", ctypes.c_int),
                ("c_planes", ctypes.c_void_p * MAX_PLANES), ("c_num_planes", ctypes.c_int), ("ldc_planes", ctypes.c_int),
                ("mask_plane", ctypes.c_void_p), ("mask_ld", ctypes.c_int), ("mask_rows", ctypes.c_int),
                ("splits", ctypes.c_int), ("workspace", ctypes.c_void_p), ("workspace_bytes", ctypes.c_size_t),
                ("a_gather", ctypes.POINTER(Gather)), ("b_gather", ctypes.POINTER(Gather)),
                ("perm_m", ctypes.c_int), ("perm_n", ctypes.c_int)]


class Conv(ctypes.Structure):
    _fields_ = [("dgrad", ctypes.c_int), ("samples", ctypes.c_int),
                ("hw_in", ctypes.c_int), ("c_in", ctypes.c_int), ("k", ctypes.c_int), ("stride", ctypes.c_int),
                ("hw_out", ctypes.c_int), ("c_out", ctypes.c_int),
                ("x", Planes), ("w", Planes), ("out", Planes),
                ("bias", ctypes.c_void_p), ("relu", ctypes.c_int),
                ("mask_plane", ctypes.c_void_p), ("mask_samples", ctypes.c_int),
                ("num_pairs", ctypes.c_int), ("pair_a", ctypes.c_int * 6), ("pair_b", ctypes.c_int * 6)]


class LearnerConfig(ctypes.Structure):
    _fields_ = [("num_envs", ctypes.c_int), ("num_steps", ctypes.c_int), ("num_actions", ctypes.c_int),
                ("conv3_filters", ctypes.c_int), ("acktr", ctypes.c_int),
                ("gamma", ctypes.c_float), ("entropy_beta", ctypes.c_float), ("value_loss_weight", ctypes.c_float),
                ("lr_start", ctypes.c_float), ("lr_end", ctypes.c_float), ("lr_decay_steps", ctypes.c_double),
                ("cov_ema_decay", ctypes.c_float), ("damping", ctypes.c_float), ("momentum", ctypes.c_float),
                ("norm_constraint", ctypes.c_float),
                ("invert_every", ctypes.c_int), ("num_cold_updates", ctypes.c_int),
                ("cold_lr", ctypes.c_float), ("cold_momentum", ctypes.c_float), ("clip_norm", ctypes.c_float),
                ("rms_decay", ctypes.c_float), ("rms_epsilon", ctypes.c_float),
                ("num_locations_mode", ctypes.c_int), ("world_size", ctypes.c_int), ("gemm_impl", ctypes.c_int),
                ("precision", ctypes.c_int), ("use_graphs", ctypes.c_int), ("conv_impl", ctypes.c_int), ("num_lanes", ctypes.c_int),
                ("seed", ctypes.c_uint64),
                ("cov_init_identity", ctypes.c_int), ("no_zero_debias", ctypes.c_int), ("inv_init_identity", ctypes.c_int)]


class MLPConfig(ctypes.Structure):
    _fields_ = [("num_envs", ctypes.c_int), ("num_steps", ctypes.c_int), ("obs_dim", ctypes.c_int),
                ("num_hidden", ctypes.c_int), ("hidden", ctypes.c_int * 4), ("num_actions", ctypes.c_int),
                ("acktr", ctypes.c_int),
                ("gamma", ctypes.c_float), ("entropy_beta", ctypes.c_float), ("value_loss_weight", ctypes.c_float),
                ("lr_start", ctypes.c_float), ("lr_end", ctypes.c_float), ("lr_decay_steps", ctypes.c_double),
                ("cov_ema_decay", ctypes.c_float), ("damping", ctypes.c_float), ("momentum", ctypes.c_float),
                ("norm_constraint", ctypes.c_float),
                ("invert_every", ctypes.c_int), ("num_cold_updates", ctypes.c_int),
                ("cold_lr", ctypes.c_float), ("cold_momentum", ctypes.c_float), ("clip_norm", ctypes.c_float),
                ("rms_decay", ctypes.c_float), ("rms_epsilon", ctypes.c_float),
                ("use_graphs", ctypes.c_int), ("seed", ctypes.c_uint64)]


# every symbol include/acx.h declares: name -> (restype, argtypes)
_P = ctypes.c_void_p
SIGNATURES = {
    "acx_last_error": (ctypes.c_char_p, []),
    "acx_version": (ctypes.c_int, []),
    "acx_launch_count": (ctypes.c_uint64, []),
    "acx_reset_launch_count": (None, []),
    "acx_preprocess_stack_u8": (ctypes.c_int, [_P, _P, _P, _P, _P, _P, _P, ctypes.c_size_t, ctypes.c_int, _P]),
    "acx_preprocess_reset_u8": (ctypes.c_int, [_P, _P, ctypes.c_size_t, ctypes.c_int, _P]),
    "acx_frame_max_u8": (ctypes.c_int, [_P, _P, _P, ctypes.c_size_t, _P]),
    "acx_framestack_push_u8": (ctypes.c_int, [_P, _P, _P, _P, ctypes.c_int, _P]),
    "acx_returns_adv": (ctypes.c_int, [_P, _P, _P, _P, ctypes.c_float, ctypes.c_int, ctypes.c_int, _P, _P, _P]),
    "acx_gemm": (ctypes.c_int, [ctypes.POINTER(Gemm), ctypes.c_int, _P]),
    "acx_gemm_workspace_bytes": (ctypes.c_size_t, [ctypes.POINTER(Gemm)]),
    "acx_split_planes": (ctypes.c_int, [_P, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_float,
                                        ctypes.POINTER(_P), ctypes.c_int, ctypes.c_int, _P]),
    "acx_debug_set_mn_desc": (None, [ctypes.c_uint32, ctypes.c_uint32, ctypes.c_uint32]),
    "acx_debug_set_fuse_reduce": (None, [ctypes.c_int]),
    "acx_obs_pairs_bf16": (ctypes.c_int, [_P, _P, ctypes.c_int, _P]),
    "acx_conv1_pairs_forward": (ctypes.c_int, [_P, ctypes.POINTER(Planes), ctypes.c_int, _P, ctypes.c_float, ctypes.POINTER(Planes),
                                               ctypes.c_int, ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int), _P]),
    "acx_debug_tc_error": (ctypes.c_int, []),
    "acx_gemm_enable_timing": (ctypes.c_int, [ctypes.c_int]),
    "acx_gemm_last_ms": (ctypes.c_int, [ctypes.POINTER(ctypes.c_float)]),
    "acx_conv_supported": (ctypes.c_int, [ctypes.POINTER(Conv)]),
    "acx_conv": (ctypes.c_int, [ctypes.POINTER(Conv), _P]),
    "acx_conv_dgrad_weights": (ctypes.c_int, [_P, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                              ctypes.c_int, ctypes.POINTER(_P), ctypes.c_int, _P]),
    "acx_debug_gemm_trace": (ctypes.c_int, [ctypes.POINTER(ctypes.c_longlong)]),
    "acx_debug_inv_trace": (ctypes.c_int, [ctypes.POINTER(ctypes.c_longlong), ctypes.c_int]),
    "acx_debug_conv_trace": (ctypes.c_int, [ctypes.POINTER(ctypes.c_longlong)]),
    "acx_learner_arena_bytes": (ctypes.c_size_t, [ctypes.POINTER(LearnerConfig)]),
    "acx_learner_create": (_P, [ctypes.POINTER(LearnerConfig), _P, ctypes.c_size_t]),
    "acx_learner_destroy": (None, [_P]),
    "acx_learner_num_params": (ctypes.c_size_t, [_P]),
    "acx_learner_set_params": (ctypes.c_int, [_P, _P, _P]),
    "acx_learner_get_params": (ctypes.c_int, [_P, _P, _P]),
    "acx_learner_refresh_weights": (ctypes.c_int, [_P, _P]),
    "acx_learner_buffer": (_P, [_P, ctypes.c_char_p, ctypes.POINTER(ctypes.c_size_t)]),
    "acx_learner_phase1": (ctypes.c_int, [_P, _P, _P, _P]),
    "acx_learner_phase2": (ctypes.c_int, [_P, _P]),
    "acx_learner_wait_input_factors": (ctypes.c_int, [_P, _P]),
    "acx_learner_update": (ctypes.c_int, [_P, _P, _P, _P]),
    "acx_learner_update_plan": (ctypes.c_int, [_P, ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int)]),
    "acx_learner_set_external_ema": (ctypes.c_int, [_P, ctypes.c_int]),
    "acx_peer_export": (ctypes.c_int, [_P, _P, ctypes.POINTER(ctypes.c_ulonglong)]),
    "acx_peer_import": (ctypes.c_void_p, [_P, ctypes.c_ulonglong]),
    "acx_learner_set_peers": (ctypes.c_int, [_P, ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_void_p)]),
    "acx_learner_wait_reduced": (ctypes.c_int, [_P, _P]),
    "acx_learner_peer_reduce_prefix": (ctypes.c_int, [_P, _P]),
    "acx_peer_error": (ctypes.c_int, []),
    "acx_learner_ema": (ctypes.c_int, [_P, _P]),
    "acx_learner_set_profiling": (ctypes.c_int, [_P, ctypes.c_int]),
    "acx_learner_stage_ms": (ctypes.c_int, [_P, ctypes.POINTER(ctypes.c_float)]),
    "acx_learner_global_step": (ctypes.c_int64, [_P]),
    "acx_learner_set_state": (ctypes.c_int, [_P, ctypes.c_int64, ctypes.c_int64, ctypes.c_int, _P]),
    "acx_learner_get_state": (ctypes.c_int, [_P, ctypes.POINTER(ctypes.c_int64), ctypes.POINTER(ctypes.c_int64),
                                             ctypes.POINTER(ctypes.c_int)]),
    "acx_learner_set_loss_weights": (ctypes.c_int, [_P, ctypes.c_float, ctypes.c_float]),
    "acx_clip_rmsprop_step": (ctypes.c_int, [_P, _P, _P, ctypes.c_size_t, ctypes.c_float, ctypes.c_float, ctypes.c_float,
                                             ctypes.c_float, _P, _P, _P]),
    "acx_clip_momentum_step": (ctypes.c_int, [_P, _P, _P, ctypes.c_size_t, ctypes.c_float, ctypes.c_float, ctypes.c_float,
                                              _P, _P, _P]),
    "acx_sample_actions": (ctypes.c_int, [_P, _P, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                          _P, _P]),
    "acx_learner_act": (ctypes.c_int, [_P, _P, ctypes.c_int, _P, ctypes.c_int, _P, _P, _P, _P]),
    "acx_mlp_arena_bytes": (ctypes.c_size_t, [ctypes.POINTER(MLPConfig)]),
    "acx_mlp_create": (_P, [ctypes.POINTER(MLPConfig), _P, ctypes.c_size_t]),
    "acx_mlp_destroy": (None, [_P]),
    "acx_mlp_num_params": (ctypes.c_size_t, [_P]),
    "acx_mlp_set_params": (ctypes.c_int, [_P, _P, _P]),
    "acx_mlp_get_params": (ctypes.c_int, [_P, _P, _P]),
    "acx_mlp_refresh_weights": (ctypes.c_int, [_P, _P]),
    "acx_mlp_buffer": (_P, [_P, ctypes.c_char_p, ctypes.POINTER(ctypes.c_size_t)]),
    "acx_mlp_update": (ctypes.c_int, [_P, _P, _P, _P]),
    "acx_mlp_set_state": (ctypes.c_int, [_P, ctypes.c_int64, ctypes.c_int64, ctypes.c_int, _P]),
    "acx_mlp_get_state": (ctypes.c_int, [_P, ctypes.POINTER(ctypes.c_int64), ctypes.POINTER(ctypes.c_int64),
                                         ctypes.POINTER(ctypes.c_int)]),
    "acx_mlp_global_step": (ctypes.c_int64, [_P]),
    "acx_mlp_act": (ctypes.c_int, [_P, _P, ctypes.c_int, _P, ctypes.c_int, _P, _P, _P, _P]),
}

_lib = None


def load():
    """Load libacx.so (building nothing: run `python __graft_entry__.py` / csrc/build.py first)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise AcxError("libacx.so not found at %s - build it with actorcritic_b200/csrc/build.py "
                       "(there is no CPU fallback)" % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    missing = []
    for name, (restype, argtypes) in SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError:
            missing.append(name)
            continue
        fn.restype = restype
        fn.argtypes = argtypes
    if missing:
        raise AcxError("libacx.so is stale or incomplete, missing symbols: %s" % ", ".join(missing))
    _lib = lib
    return lib


def check(status):
    if status != 0:
        raise AcxError(load().acx_last_error().decode("utf-8", "replace"))


def launch_count():
    return int(load().acx_launch_count())
