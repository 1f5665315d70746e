"""ctypes binding of libhgru_b200.so (include/hgru_b200.h).  No torch types cross the boundary:
tensors are passed as raw device / host pointers plus the CUDA stream handle.

There is no CPU fallback: if the shared library is missing this module raises at import of the
symbol table, and every compute call needs a CUDA device."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libhgru_b200.so")

MODE_FP32 = 0
MODE_BF16 = 1
MODE_BF16X3 = 2
MODE_FP16 = 3
MODES = {"fp32": MODE_FP32, "bf16": MODE_BF16, "bf16x3": MODE_BF16X3, "fp16": MODE_FP16}

HGRU_PARAM_ORDER = ("p_r", "i_r", "i_b", "o_r", "o_b", "beta", "nu", "gamma", "kappa", "omega",
                    "rho", "lateral_bias")

_c_float_p = ctypes.c_void_p      # raw addresses (device or host)


class PoseParams(ctypes.Structure):
    """pose_params_t of include/hgru_b200.h (same field order)."""
    _fields_ = ([(n, ctypes.c_void_p) for n in (
        "conv_1_filters", "conv_1_biases", "conv_2_filters", "conv_2_biases",
        "conv_3_filters", "conv_3_biases", "fc_1_weights", "fc_1_biases",
        "fc_out_weights", "fc_out_biases")]
        + [("bn", (ctypes.c_void_p * 4) * 5)]
        + [(n, ctypes.c_void_p) for n in HGRU_PARAM_ORDER])


class AttnParams(ctypes.Structure):
    """attn_params_t of include/hgru_b200.h (same field order)."""
    _fields_ = [("conv_filters", ctypes.c_void_p * 5), ("conv_biases", ctypes.c_void_p * 5),
                ("fc_1_weights", ctypes.c_void_p), ("fc_1_biases", ctypes.c_void_p),
                ("fc_out_weights", ctypes.c_void_p), ("fc_out_biases", ctypes.c_void_p),
                ("bn", (ctypes.c_void_p * 4) * 6)]


# every symbol include/hgru_b200.h declares: name -> (restype, argtypes)
_P = ctypes.c_void_p
_I = ctypes.c_int
SIGNATURES = {
    "hgru_last_error": (ctypes.c_char_p, []),
    "hgru_version": (_I, []),
    "hgru_plan_create": (_I, [_I, _I, _I, _I, _I, _I, _I, ctypes.POINTER(_P)]),
    "hgru_plan_destroy": (_I, [_P]),
    "hgru_set_params": (_I, [_P] + [_P] * 12 + [_P]),
    "hgru_forward": (_I, [_P, _P, _P, _P, _P, _P, _P]),
    "hgru_forward_batch": (_I, [_P, _I, _P, _P, _P, _P, _P, _P]),
    "hgru_plan_workspace_bytes": (ctypes.c_size_t, [_P]),
    "hgru_plan_launch_count": (_I, [_P]),
    "pose_plan_create": (_I, [_I, _I, _I, _I, _I, _I, _I, _I, ctypes.POINTER(_P)]),
    "pose_plan_destroy": (_I, [_P]),
    "pose_set_params": (_I, [_P, ctypes.POINTER(PoseParams), ctypes.c_float, _P]),
    "pose_forward": (_I, [_P, _P, _P, _P, _P]),
    "pose_forward_host": (_I, [_P, _P, _P, _P, _P]),
    "pose_forward_batch": (_I, [_P, _I, _P, _P, _P, _P]),
    "pose_forward_host_batch": (_I, [_P, _I, _P, _P, _P, _P]),
    "pose_set_hidden_init": (_I, [_P, _I]),
    "pose_get_activation": (_I, [_P, ctypes.c_char_p, _P, _P]),
    "pose_plan_workspace_bytes": (ctypes.c_size_t, [_P]),
    "pose_plan_launch_count": (_I, [_P]),
    "hgru_enable_kernel_timing": (_I, [_I]),
    "pose_plan_kernel_times": (_I, [_P, ctypes.POINTER(ctypes.c_float), ctypes.POINTER(_I)]),
    "pose_plan_sm_clock_ghz": (_I, [_P, ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_float)]),
    "layer_conv2d_forward": (_I, [_P, _I, _I, _I, _I, _P, _I, _I, _P, _I, _P, _P]),
    "circuit_gate_forward": (_I, [_P, ctypes.c_size_t, _I, _P, _P, _P, _P, _P]),
    "circuit_input_integration_forward": (_I, [_P, _P, _P, _P, _P, ctypes.c_float, ctypes.c_size_t, _I, _P, _P]),
    "circuit_output_integration_forward": (_I, [_P, _P, _P, _P, _P, _P, _P, ctypes.c_float, _P, ctypes.c_size_t, _I,
                                                _P, _P]),
    "layer_max_pool2x2_forward": (_I, [_P, _I, _I, _I, _I, _P, _P]),
    "layer_pool_same_forward": (_I, [_P, _I, _I, _I, _I, _I, _I, _P, _P]),
    "layer_batchnorm_moments0_forward": (_I, [_P, _I, ctypes.c_size_t, ctypes.c_float, _P, _P]),
    "layer_fc_forward": (_I, [_P, _I, _I, _P, _P, _I, _P, _P]),
    "layer_resize_bilinear_forward": (_I, [_P, _I, _I, _I, _I, _I, _P, _P]),
    "layer_batch_norm_forward": (_I, [_P, ctypes.c_size_t, _I, _P, _P, _P, _P, ctypes.c_float, _I, _I, ctypes.c_float,
                                      ctypes.c_ulonglong, ctypes.c_float, _P, _P, _P, _P, _P]),
    "crop_area3d_forward": (_I, [_P, _I, _I, _I, ctypes.c_float, _P, _P, ctypes.c_float, ctypes.c_double, _P,
                                 _I, _I, _P]),
    "depth_preprocess_forward": (_I, [_P, ctypes.c_size_t, ctypes.c_uint, ctypes.c_uint, ctypes.c_double,
                                      ctypes.c_double, _P, _P]),
    "crop_windows_forward": (_I, [_P, _P, ctypes.c_double, ctypes.c_double, ctypes.c_double, _I, _I, _I, _I, _I,
                                  ctypes.c_double, ctypes.c_double, ctypes.c_double, ctypes.c_double, ctypes.c_double,
                                  _P, _P, _P, _P, _P, _P]),
    "calculate_com_workspace_bytes": (ctypes.c_size_t, [_I, ctypes.c_longlong]),
    "calculate_com_forward": (_I, [_P, _I, _I, _I, ctypes.c_float, ctypes.c_float, ctypes.c_float, _P, _P,
                                   ctypes.c_longlong, _P, _P, _P, _P]),
    "pose_postprocess_forward": (_I, [_P, _P, _I, _I, ctypes.c_double, ctypes.c_double, ctypes.c_double,
                                      ctypes.c_double, ctypes.c_float, _P, _P, _P]),
    "joint_error_forward": (_I, [_P, _P, _I, _I, _P, _P, _P, _P]),
    "joint_error_stats_forward": (_I, [_P, _P, _I, _I, _I, _P, _P, _P, _P, _P, _P]),
    "joint_error_count_within_forward": (_I, [_P, _I, ctypes.c_float, _P, _P]),
    "axis1_error_mean_forward": (_I, [_P, _P, _I, _I, _I, _I, _P, _P, _P]),
    "attn_plan_create": (_I, [_I, _I, _I, ctypes.POINTER(_I), _I, _I, ctypes.POINTER(_P)]),
    "attn_plan_create_mode": (_I, [_I, _I, _I, ctypes.POINTER(_I), _I, _I, _I, ctypes.POINTER(_P)]),
    "attn_plan_destroy": (_I, [_P]),
    "attn_set_params": (_I, [_P, ctypes.POINTER(AttnParams), ctypes.c_float, _P]),
    "attn_forward": (_I, [_P, _P, _P, _P]),
    "attn_forward_batch": (_I, [_P, _I, _P, _P, _P]),
    "attn_get_activation": (_I, [_P, ctypes.c_char_p, _P, _P]),
    "attn_plan_workspace_bytes": (ctypes.c_size_t, [_P]),
    "attn_plan_launch_count": (_I, [_P]),
}

_lib = None


def load():
    """Load the shared library (once) and type its entry points.  Fails loudly when it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "libhgru_b200.so is not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -C monkey-pose_b200/csrc` (needs nvcc, sm_100a). There is no CPU fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the export is missing
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


class HgruError(RuntimeError):
    pass


def check(rc, what):
    if rc != 0:
        msg = load().hgru_last_error()
        text = msg.decode() if msg else ""
        if rc == 2:
            raise NotImplementedError("%s: %s" % (what, text))
        if rc == 1:
            raise ValueError("%s: %s" % (what, text))
        raise HgruError("%s failed (code %d): %s" % (what, rc, text))
