"""ctypes binding of the C ABI declared in include/spectral_conv_b200.h.

There is no fallback: if the shared object is missing or a symbol is absent, importing the binding
raises, and every product entry point above it fails with it.
"""
import ctypes
import os
import threading

from .build import LIB_PATH

SC_MAX_DIMS = 4
NORMS = {"forward": 0, "backward": 1, "ortho": 2}
FLAG_RESAMPLE = 1
FLAG_GRID_F16, FLAG_GRID_BF16 = 2, 4     # x / dx stored as float16 / bfloat16
ACT_IDENTITY, ACT_GELU, ACT_RELU, ACT_SILU, ACT_TANH = 0, 1, 2, 3, 4
POINTWISE_TANH, POINTWISE_TANH_BACKWARD, POINTWISE_ROUND_HALF, POINTWISE_ADD_I_TIMES, POINTWISE_MUL_NEG_I, POINTWISE_MUL = 0, 1, 2, 3, 4, 5

c_void_p = ctypes.c_void_p
c_int = ctypes.c_int
c_i32 = ctypes.c_int32
c_i64 = ctypes.c_int64
c_size_t = ctypes.c_size_t


class ScProblem(ctypes.Structure):
    _fields_ = [
        ("ndim", c_i32),
        ("grid", c_i32 * SC_MAX_DIMS),
        ("out_grid", c_i32 * SC_MAX_DIMS),
        ("n_modes", c_i32 * SC_MAX_DIMS),
        ("max_n_modes", c_i32 * SC_MAX_DIMS),
        ("fft_norm", c_i32),
        ("flags", c_i32),
    ]


# name -> (restype, argtypes); mirrors include/spectral_conv_b200.h one to one
SIGNATURES = {
    "sc_plan_create": (c_int, [ctypes.POINTER(ScProblem), ctypes.POINTER(c_void_p)]),
    "sc_plan_destroy": (None, [c_void_p]),
    "sc_plan_kept_modes": (c_int, [c_void_p, ctypes.POINTER(c_i32)]),
    "sc_plan_mode_bins": (c_int, [c_void_p, c_int, ctypes.POINTER(c_i32), ctypes.POINTER(c_i32)]),
    "sc_workspace_bytes": (c_size_t, [c_void_p, c_i64]),
    "sc_plan_set_fast_path": (c_int, [c_void_p, c_int]),
    "sc_plan_uses_fast_path": (c_int, [c_void_p]),
    "sc_plan_set_reserved_sms": (c_int, [c_void_p, c_int]),
    "sc_analyze": (c_int, [c_void_p, c_void_p, c_i64, c_void_p, c_int, c_void_p, c_size_t, c_void_p]),
    "sc_synthesize": (c_int, [c_void_p, c_void_p, c_i64, c_i32, c_void_p, c_void_p, c_int, c_void_p, c_size_t,
                              c_void_p]),
    "sc_contract_dense": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_i32, c_i32, c_i32, c_void_p]),
    "sc_contract_dense_backward": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                           c_i32, c_i32, c_i32, c_void_p]),
    "sc_bias_grad": (c_int, [c_void_p, c_void_p, c_void_p, c_i32, c_i32, c_void_p]),
    "sc_forward_dense": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, ctypes.POINTER(c_i32), c_i32, c_i32,
                                 c_i32, c_void_p, c_size_t, c_void_p]),
    "sc_backward_dense": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_i32, c_void_p, c_void_p, c_void_p, c_i32, c_i32,
                                  c_i32, c_void_p, c_size_t, c_void_p, c_void_p]),
    "sc_tucker_saved_elems": (c_size_t, [c_void_p, c_i32, c_i32, c_i32, c_void_p]),
    "sc_tucker_workspace_bytes": (c_size_t, [c_void_p, c_i32, c_i32, c_i32, c_void_p]),
    "sc_forward_tucker": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                  c_i32, c_i32, c_i32, c_void_p, c_void_p, c_size_t, c_void_p]),
    "sc_backward_tucker": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                   c_void_p, c_void_p, c_void_p, c_void_p, c_i32, c_i32, c_i32, c_void_p, c_void_p, c_size_t, c_void_p]),
    "sc_cp_saved_elems": (c_size_t, [c_void_p, c_i32, c_i32, c_i32, c_i32]),
    "sc_cp_workspace_bytes": (c_size_t, [c_void_p, c_i32, c_i32, c_i32, c_i32]),
    "sc_forward_cp": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                              c_i32, c_i32, c_i32, c_i32, c_void_p, c_size_t, c_void_p]),
    "sc_backward_cp": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                               c_void_p, c_void_p, c_void_p, c_i32, c_i32, c_i32, c_i32, c_void_p, c_size_t, c_void_p]),
    "sc_tt_saved_elems": (c_size_t, [c_void_p, c_i32, c_i32, c_i32, c_void_p]),
    "sc_tt_workspace_bytes": (c_size_t, [c_void_p, c_i32, c_i32, c_i32, c_void_p]),
    "sc_forward_tt": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                              c_i32, c_i32, c_i32, c_void_p, c_void_p, c_size_t, c_void_p]),
    "sc_backward_tt": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                               c_void_p, c_void_p, c_i32, c_i32, c_i32, c_void_p, c_void_p, c_size_t, c_void_p]),
    "sc_allreduce_p2p": (c_int, [c_void_p, c_void_p, c_i32, c_i32, c_i64, ctypes.c_float, c_i32, c_void_p]),
    "sc_event_create": (c_int, [ctypes.POINTER(c_void_p)]),
    "sc_event_destroy": (None, [c_void_p]),
    "sc_stream_wait_event": (c_int, [c_void_p, c_void_p]),
    "sc_table_contract": (c_int, [c_void_p, c_i64, c_i64, c_int, c_void_p, c_void_p, c_i64, c_i32, c_i32, c_i32, c_void_p]),
    "sc_pair_reduce": (c_int, [c_void_p, c_void_p, c_void_p, c_i64, c_i64, c_i64, c_i32, c_i32, c_i32, c_void_p]),
    "sc_problem_table": (c_int, [c_void_p, c_int, c_int, c_void_p, ctypes.c_size_t, c_void_p, c_void_p]),
    "sc_problem_mode_bins": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p]),
    "sc_cp_scale": (c_int, [c_void_p, c_void_p, c_i32, c_void_p, c_void_p, c_i32, c_void_p]),
    "sc_cp_apply": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_i32, c_i64, c_void_p]),
    "sc_cp_dscale": (c_int, [c_void_p, c_void_p, c_void_p, c_i32, c_i64, c_void_p]),
    "sc_cp_factor_grad": (c_int, [c_void_p, c_void_p, c_i32, c_void_p, c_void_p, c_void_p, c_i32, c_i32, c_void_p]),
    "sc_channel_mix": (c_int, [c_void_p, c_void_p, c_i64, c_i64, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p,
                               c_i32, c_i32, c_i32, c_i64, c_void_p]),
    "sc_channel_mix_act_backward": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                            c_i32, c_i32, c_i64, c_void_p]),
    "sc_channel_mix_weight_grad": (c_int, [c_void_p, c_void_p, c_void_p, c_i32, c_i32, c_i32, c_i64, c_void_p]),
    "sc_pointwise": (c_int, [c_int, c_void_p, c_void_p, c_void_p, c_i64, c_void_p]),
    "sc_layer_set_tensor_cores": (c_int, [c_int]),
    "sc_layer_uses_tensor_cores": (c_int, []),
    # host checks of the layer kernels' tile functions (tests only)
    "sc_hostcheck_channel_mix": (c_int, [c_void_p, c_void_p, c_i64, c_i64, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p,
                                         c_void_p, c_i32, c_i32, c_i32, c_i64]),
    "sc_hostcheck_channel_mix_act_backward": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                                      c_void_p, c_i32, c_i32, c_i64]),
    "sc_hostcheck_channel_mix_weight_grad": (c_int, [c_void_p, c_void_p, c_void_p, c_i32, c_i32, c_i32, c_i64]),
    "sc_hostcheck_pointwise": (c_int, [c_int, c_void_p, c_void_p, c_void_p, c_i64]),
    "sc_hostcheck_convert": (c_int, [c_int, c_int, c_void_p, c_void_p, c_i64]),
    "sc_hostcheck_chain_log": (c_int, [c_void_p, c_int, c_int, c_i32, c_i32, c_i32, c_void_p, c_void_p, c_size_t, c_void_p]),
    "sc_probe_tma_gather": (c_int, [c_void_p, c_i32, c_i32, c_i64, c_void_p, c_void_p]),
    "sc_last_error": (ctypes.c_char_p, []),
    "sc_kernel_launch_count": (ctypes.c_uint64, []),
    "sc_build_info": (ctypes.c_char_p, []),
    "sc_selftest_umma": (c_int, [c_void_p, c_void_p, c_void_p, c_i32, c_i32, c_void_p]),
    "sc_selftest_umma_ts": (c_int, [c_void_p, c_void_p, c_void_p, c_i32, c_i32, c_void_p]),
}

_lock = threading.Lock()
_lib = None


def load():
    """Loads libspectral_conv_b200.so (built in-tree by `neuraloperator_b200.build`). Raises if absent."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.isfile(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: the CUDA extension was not built. Run `python -m neuraloperator_b200.build` "
                "(or __graft_entry__.build()). neuraloperator_b200 has no CPU or PyTorch fallback.")
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)   # AttributeError if the .so does not export it
            fn.restype = res
            fn.argtypes = args
        _lib = lib
        return lib


def check(rc, what):
    if rc != 0:
        msg = load().sc_last_error()
        raise RuntimeError(f"{what} failed: {msg.decode() if msg else 'unknown error'}")


def launch_count():
    return int(load().sc_kernel_launch_count())
