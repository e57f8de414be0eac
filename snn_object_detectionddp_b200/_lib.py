"""ctypes binding of libsnnb200.so (C ABI in include/snn_b200.h).

There is NO fallback: if the shared library is missing or a call fails, an exception is raised.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libsnnb200.so")

GEOM_3x3_S1, GEOM_3x3_S2, GEOM_1x1, GEOM_T2x2_S2 = 0, 1, 2, 3
ACT_LIF, ACT_SILU = 0, 1
GEOM_TAPS = {GEOM_3x3_S1: 9, GEOM_3x3_S2: 9, GEOM_1x1: 1, GEOM_T2x2_S2: 4}

_c = ctypes
_P, _I, _L, _F, _D = _c.c_void_p, _c.c_int, _c.c_longlong, _c.c_float, _c.c_double

_SIGNATURES = {
    "snn_conv_fprop": [_I, _I, _I, _I, _P, _I, _L, _P, _I, _L, _P, _I, _I, _I, _I, _I, _P, _P, _I, _L, _I, _I, _P],
    "snn_conv_fprop_stats": [_I, _I, _I, _I, _P, _I, _L, _P, _I, _L, _P, _I, _I, _I, _I, _I, _P, _I, _P, _P],
    "snn_bn_stats_from_partials": [_P, _P, _I, _I, _I, _P],
    "snn_bn_finalize_partials": [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _F, _F, _P],
    "snn_conv_dgrad": [_I, _I, _I, _I, _P, _I, _L, _P, _I, _I, _I, _P, _I, _L, _I, _I, _P],
    "snn_conv_wgrad": [_I, _I, _I, _I, _P, _I, _L, _P, _I, _L, _P, _I, _I, _P],
    "snn_weight_prep": [_P, _P, _P, _I, _I, _I, _P],
    "snn_bn_stats": [_P, _P, _P, _I, _I, _I, _P],
    "snn_bn_finalize": [_P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _F, _F, _I, _P],
    "snn_bn_act_fwd": [_I, _P, _P, _P, _P, _P, _P, _P, _I, _L, _I, _I, _F, _F, _P],
    "snn_bn_act_fwd_count": [_P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _L, _I, _I, _F, _F, _P],
    "snn_bn_act_bwd": [_I, _I, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _F, _F, _F, _P],
    "snn_bn_act_bwd2": [_I, _I, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _F, _F, _F, _P],
    "snn_bn_act_bwd2_ds": [_I, _I, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _F, _F, _F, _P, _P],
    "snn_spike_reg_coef": [_P, _P, _I, _I, _D, _D, _D, _D, _D, _P, _P, _P, _I, _I, _P],
    "snn_bn_bwd_dx": [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _P],
    "snn_lstm_gates_fwd": [_P, _P, _P, _P, _P, _L, _I, _P],
    "snn_lstm_gates_bwd": [_P, _P, _P, _P, _P, _P, _P, _P, _L, _I, _P],
    "snn_nchw_to_nhwc": [_P, _P, _I, _I, _I, _I, _L, _I, _P],
    "snn_nhwc_to_nchw": [_P, _I, _P, _I, _I, _I, _L, _I, _P],
    "snn_colsum_bf16": [_P, _P, _L, _I, _P],
    "snn_bilinear_resize": [_I, _P, _P, _I, _I, _I, _I, _I, _I, _P],
    "snn_nhwc_pad_crop": [_P, _P, _I, _I, _I, _I, _I, _I, _P],
    "snn_dw3x3_fprop": [_P, _P, _P, _I, _I, _I, _I, _P],
    "snn_dw3x3_fprop_stats": [_P, _P, _P, _I, _I, _I, _I, _I, _P, _P],
    "snn_dw3x3_dgrad": [_P, _P, _P, _I, _I, _I, _I, _P],
    "snn_dw3x3_wgrad": [_P, _P, _P, _I, _I, _I, _I, _P],
    "snn_space_to_depth8": [_P, _P, _I, _I, _I, _I, _P],
    "snn_space_to_depth8_u8": [_P, _P, _I, _I, _I, _I, _P],
    "snn_detect_decode": [_P, _P, _P, _P, _I, _I, _I, _I, _I, _P, _P, _P],
    "snn_detect_loss_fwd": [_P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _P, _P],
    "snn_detect_loss_bwd": [_P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _P, _P, _P, _P],
    "snn_detect_assign_loss_fwd": [_P, _P, _I, _P, _P, _P, _P, _P, _P, _F, _F, _I, _I, _I, _I, _I, _I, _P, _P, _P, _P, _P, _P, _P, _P,
                                   _P, _P, _P, _P],
    "snn_tal_assign": [_P, _P, _P, _P, _P, _P, _P, _F, _F, _I, _I, _I, _I, _I, _P, _P, _P, _P, _P],
    "snn_detect_loss_bwd_rows": [_P, _P, _I, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _P, _P, _P, _P, _I, _P],
    "snn_nms": [_P, _I, _I, _I, _F, _F, _I, _I, _I, _I, _F, _P, _L, _P, _P, _P, _P],
    "snn_det_match": [_P, _P, _I, _I, _P, _P, _P, _I, _F, _F, _P, _I, _P, _P, _P, _P, _L, _P, _P, _P, _P, _P],
    "snn_det_metrics_finalize": [_P, _P, _P, _L, _P, _I, _P, _P, _P, _P],
    "snn_grad_sumsq": [_P, _L, _P, _I, _P],
    "snn_adamw_step": [_P, _P, _P, _P, _P, _L, _P, _P, _P, _P, _I, _I, _P],
    "snn_ema_update": [_P, _P, _L, _P, _I, _P, _P, _I, _P],
}

_lib = None
launch_count = 0  # number of libsnnb200 kernel-launching calls made (bench.py reports it)


class SnnKernelError(RuntimeError):
    pass


def exported_symbols():
    return sorted(list(_SIGNATURES) + ["snn_last_error", "snn_version", "snn_debug_set", "snn_set_tile_scheduling", "snn_set_dependent_launch", "snn_get_dependent_launch", "snn_set_deterministic", "snn_get_deterministic", "snn_conv_plan", "snn_tensor_map_cache_stats", "snn_conv_stats_groups", "snn_bn_stats_workspace_floats", "snn_nms_workspace_keys",
                                             "snn_tal_workspace_bytes", "snn_dw3x3_stats_blocks", "snn_bn_finalize_workspace_doubles"])


def lib():
    """Load libsnnb200.so (once). Raises if it was not built: the product has no CPU path."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise SnnKernelError(
                f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a). There is no fallback path.")
        L = ctypes.CDLL(LIB_PATH)
        for name, args in _SIGNATURES.items():
            fn = getattr(L, name)
            fn.argtypes = args
            fn.restype = _I
        L.snn_last_error.restype = ctypes.c_char_p
        L.snn_version.restype = _I
        L.snn_conv_stats_groups.argtypes = [_I, _I, _I, _I, _I, ctypes.POINTER(_I)]
        L.snn_conv_stats_groups.restype = _L
        L.snn_bn_stats_workspace_floats.argtypes = [_I, _I, _I]
        L.snn_bn_stats_workspace_floats.restype = _L
        L.snn_nms_workspace_keys.argtypes = [_I, _I, _I]
        L.snn_nms_workspace_keys.restype = _L
        L.snn_bn_finalize_workspace_doubles.argtypes = [_I, _I, _I]
        L.snn_bn_finalize_workspace_doubles.restype = _L
        L.snn_dw3x3_stats_blocks.argtypes = [_I, _I, _I]
        L.snn_dw3x3_stats_blocks.restype = _L
        L.snn_tal_workspace_bytes.argtypes = [_I, _I, _I]
        L.snn_tal_workspace_bytes.restype = _L
        L.snn_debug_set.argtypes = [_I, _I]
        L.snn_debug_set.restype = None
        if "SNN_WGRAD_STRIP" in os.environ:        # A/B timing: 1 = tap-by-tap wgrad
            L.snn_debug_set(13, int(os.environ["SNN_WGRAD_STRIP"]))
        if "SNN_WGRAD_ROUNDS" in os.environ:
            L.snn_debug_set(14, int(os.environ["SNN_WGRAD_ROUNDS"]))
        if "SNN_ROW_STRIP" in os.environ:          # A/B timing: 1 = row-strip mode off, 2 = not for 256-column tiles
            L.snn_debug_set(12, int(os.environ["SNN_ROW_STRIP"]))
        L.snn_set_tile_scheduling.argtypes = [_I]
        L.snn_set_tile_scheduling.restype = None
        L.snn_set_dependent_launch.argtypes = [_I]
        L.snn_set_dependent_launch.restype = None
        L.snn_get_dependent_launch.argtypes = []
        L.snn_get_dependent_launch.restype = _I
        L.snn_set_dependent_launch(int(os.environ.get("SNN_DEPENDENT_LAUNCH", "0")))
        L.snn_conv_plan.argtypes = [_I] * 10 + [ctypes.POINTER(_I)]
        L.snn_conv_plan.restype = _I
        L.snn_set_deterministic.argtypes = [_I]
        L.snn_set_deterministic.restype = None
        L.snn_get_deterministic.argtypes = []
        L.snn_get_deterministic.restype = _I
        L.snn_set_deterministic(int(os.environ.get("SNN_DETERMINISTIC", "0")))
        L.snn_tensor_map_cache_stats.argtypes = [ctypes.POINTER(ctypes.c_ulonglong), ctypes.POINTER(ctypes.c_ulonglong)]
        L.snn_tensor_map_cache_stats.restype = None
        _lib = L
    return _lib


def ptr(t):
    """Device pointer of a tensor (or None -> NULL)."""
    if t is None:
        return None
    return t.data_ptr()


_call_dev = None   # device of the tensors of the call being prepared (set by require_cuda at the top of every wrapper)


def stream_ptr():
    """Current stream of the device the call's tensors live on (NOT of torch's current device: the reference does
    `model.to('cuda:3')` without ever calling set_device, main.py:120-131)."""
    return torch.cuda.current_stream(_call_dev).cuda_stream


profile = None    # when set to a list, every call is bracketed by CUDA events: (name, work, ev_start, ev_end)
trace = None      # when set to a list, every call appends (name, work): the launch sequence of a step (bench.py matches it
                  # against the CUPTI kernel records of a replayed CUDA graph)


def call(name, *args, work=None):
    """Invoke one ABI entry point on the stream of the tensors' device.  `work` = ("flop" | "byte", amount) is the
    algorithmic work of this launch (used by bench.py's live roofline accounting; ignored otherwise)."""
    global launch_count
    dev = _call_dev
    if profile is not None:
        e0 = torch.cuda.Event(enable_timing=True)
        e0.record(torch.cuda.current_stream(dev))
    fn = getattr(lib(), name)
    if dev is not None and dev.index is not None and dev.index != torch.cuda.current_device():
        with torch.cuda.device(dev):          # kernels launch in the CURRENT context: make it the tensors' device
            rc = fn(*args)
    else:
        rc = fn(*args)
    if rc != 0:
        raise SnnKernelError(f"{name} failed (rc={rc}): {lib().snn_last_error().decode()}")
    launch_count += 1
    if trace is not None:
        trace.append((name, work))
    if profile is not None:
        e1 = torch.cuda.Event(enable_timing=True)
        e1.record(torch.cuda.current_stream(dev))
        profile.append((name, work, e0, e1))


def require_cuda(*tensors):
    """Every tensor of a call must be a CUDA tensor on ONE device; that device becomes the launch device."""
    global _call_dev
    dev = None
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise SnnKernelError("snn_object_detectionddp_b200 kernels run on CUDA tensors only (no CPU fallback)")
        if dev is None:
            dev = t.device
        elif t.device != dev:
            raise SnnKernelError(f"tensors of one kernel call live on different devices ({dev} vs {t.device})")
    _call_dev = dev
    return dev
