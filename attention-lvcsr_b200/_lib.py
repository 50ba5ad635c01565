"""ctypes binding of csrc/liblvsr_b200.so -- the C ABI declared in include/lvsr_b200.h.

There is NO fallback: if the shared library is missing, importing the package works
(so host-only logic can be unit-tested) but any compute call raises.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# LVSR_B200_LIB: load another build of the same library (A/B measurements of kernel variants on one box)
LIB_PATH = os.environ.get("LVSR_B200_LIB") or os.path.join(_HERE, "csrc", "liblvsr_b200.so")

LVSR_MAX_LAYERS = 8
NORMALIZERS = {"softmax": 0, "logistic": 1, "relu": 2}
ACTIVATIONS = {"maxout": 0, "relu": 1, "tanh": 2, "identity": 3}
PRIORS = {"expanding": 0, "window_around_mean": 1, "window_around_median": 2}


class LvsrConfig(C.Structure):
    """Mirror of ``lvsr_config`` (include/lvsr_b200.h)."""
    _fields_ = [
        ("num_features", C.c_int32),
        ("num_layers", C.c_int32),
        ("dims_bidir", C.c_int32 * LVSR_MAX_LAYERS),
        ("subsample", C.c_int32 * LVSR_MAX_LAYERS),
        ("dim_dec", C.c_int32),
        ("dim_matcher", C.c_int32),
        ("conv_n", C.c_int32),
        ("conv_num_filters", C.c_int32),
        ("num_phonemes", C.c_int32),
        ("dim_feedback", C.c_int32),
        ("post_merge_dim", C.c_int32),
        ("maxout_pieces", C.c_int32),
        ("post_merge_activation", C.c_int32),
        ("use_states_for_readout", C.c_int32),
        ("energy_normalizer", C.c_int32),
        ("prior_type", C.c_int32),
        ("prior_initial_begin", C.c_double),
        ("prior_initial_end", C.c_double),
        ("prior_min_speed", C.c_double),
        ("prior_max_speed", C.c_double),
        ("prior_before", C.c_double),
        ("prior_after", C.c_double),
        ("one_of_n_feedback", C.c_int32),
        ("reserved", C.c_int32),
    ]


class LvsrTrainConfig(C.Structure):
    """Mirror of ``lvsr_train_config`` (include/lvsr_b200.h)."""
    _fields_ = [("gradient_threshold", C.c_float), ("use_momentum", C.c_int32), ("scale", C.c_float),
                ("momentum", C.c_float), ("use_adadelta", C.c_int32), ("decay_rate", C.c_float),
                ("epsilon", C.c_float), ("max_norm", C.c_float), ("burn_in_steps", C.c_int32), ("decay", C.c_float)]


# name -> (restype, argtypes); every symbol include/lvsr_b200.h declares
_P = C.c_void_p
_I = C.c_int32
SIGNATURES = {
    "lvsr_last_error": (C.c_char_p, []),
    "lvsr_version": (C.c_int, []),
    "lvsr_model_create": (C.c_int, [C.POINTER(LvsrConfig), C.POINTER(_P)]),
    "lvsr_model_destroy": (C.c_int, [_P]),
    "lvsr_model_num_params": (C.c_int, [_P]),
    "lvsr_model_param_name": (C.c_char_p, [_P, C.c_int]),
    "lvsr_model_param_shape": (C.c_int, [_P, C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_int32)]),
    "lvsr_model_set_param": (C.c_int, [_P, C.c_char_p, _P, C.c_int64]),
    "lvsr_model_get_param": (C.c_int, [_P, C.c_char_p, _P, C.c_int64]),
    "lvsr_model_flat_size": (C.c_int64, [_P]),
    "lvsr_model_param_offset": (C.c_int, [_P, C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "lvsr_model_flat_params": (C.c_void_p, [_P]),
    "lvsr_model_finalize": (C.c_int, [_P]),
    "lvsr_model_status": (C.c_int, [_P, C.POINTER(C.c_int32), C.POINTER(C.c_int64)]),
    "lvsr_dec_scan_plan": (C.c_int, [C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "lvsr_encoded_length": (C.c_int, [_P, _I]),
    "lvsr_encoded_dim": (C.c_int, [_P]),
    "lvsr_encoder_forward": (C.c_int, [_P, _P, _P, _I, _I, _P, _P, _P]),
    "lvsr_preprocess": (C.c_int, [_P, _P, _I, _I, _P, _P]),
    "lvsr_cost_matrix": (C.c_int, [_P, _P, _P, _I, _I, _P, _P, _I, _P, _P, _P, _P, _P, _P]),
    "lvsr_initial_states": (C.c_int, [_P, _I, _I, _P, _P, _P, _P, _P, _P, _P]),
    "lvsr_logprobs": (C.c_int, [_P, _P, _P, _P, _I, _I, _P, _I, _P, _P, _P, _P, _P]),
    "lvsr_next_states": (C.c_int, [_P, _P, _P, _P, _I, _I, _P, _I, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "lvsr_search_expand": (C.c_int, [_P, _P, _P, _P, _I, _I, _P, _P, _P, _P, _I, _I, _P, _P, _P, _P, _I, _P, _P, _P, _P, _P, _P, _P, _P]),
    "lvsr_search_advance": (C.c_int, [_P, _P, _P, _P, _I, _I, _P, _I, _P, _P, _P, _P, _P, _I, _P, _P, _P, _P, _P, _P, _I,
                                      _P, _P, _P, _P, _P, _P]),
    "lvsr_beam_search_many": (C.c_int, [_P, _P, _P, _P, _I, _I, _P, _P, _I, _I, _I, C.c_double, C.c_double, _I, C.POINTER(_P), _P]),
    "lvsr_search_result_count": (C.c_int, [_P, _I]),
    "lvsr_search_result_length": (C.c_int, [_P, _I, _I]),
    "lvsr_search_result_get": (C.c_int, [_P, _I, _I, _P, _P]),
    "lvsr_search_result_destroy": (C.c_int, [_P]),
    "lvsr_recognizer_cost_host": (C.c_int, [_P, _P, _P, _P, _P, _I, _I, _I, _P, _P]),
    "lvsr_train_cost_and_grads": (C.c_int, [_P, _P, _P, _P, _P, _I, _I, _I, C.c_float, _P, _P, _P]),
    "lvsr_train_apply_updates": (C.c_int, [_P, _P, C.c_float, C.POINTER(LvsrTrainConfig), _P]),
    "lvsr_train_gradient_norm": (C.c_int, [_P, C.POINTER(C.c_float)]),
    "lvsr_train_reset": (C.c_int, [_P]),
    "lvsr_launch_count": (C.c_int64, [C.c_int]),
    "lvsr_profile_enable": (C.c_int, [C.c_int]),
    "lvsr_profile_read": (C.c_int, [C.c_char_p, C.POINTER(C.c_double), C.POINTER(C.c_int64)]),
}

_lib = None


def load():
    """Load the shared library (once) and declare every signature."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "%s is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(attention-lvcsr_b200 has no CPU or PyTorch fallback)" % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if a declared symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        msg = load().lvsr_last_error()
        raise RuntimeError("lvsr_b200: " + (msg.decode("utf-8", "replace") if msg else "error %d" % rc))
