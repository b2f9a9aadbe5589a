"""ctypes binding of libbnnchaos.so (the C ABI declared in include/bnnchaos.h).

The shared library is built in-tree by ``__graft_entry__.build()`` (or ``make -C
bnn_chaos_model_b200/csrc``).  There is no CPU or PyTorch-eager fallback: if the library is
missing, or an entry point reports an error, the caller gets an exception.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# BNN_CHAOS_LIB selects a diagnostic build of the same library (e.g. libbnnchaos_tl.so); there is no other backend
LIB_PATH = os.environ.get("BNN_CHAOS_LIB") or os.path.join(_HERE, "libbnnchaos.so")

c_f32p = C.c_void_p  # device / host float* (passed as integers from tensor.data_ptr())
c_i32p = C.c_void_p


class ModelConfig(C.Structure):
    """bnn_model_config (include/bnnchaos.h)."""

    _fields_ = [
        ("n_features", C.c_int32),
        ("hidden", C.c_int32),
        ("latent", C.c_int32),
        ("n_in_layers", C.c_int32),
        ("n_out_layers", C.c_int32),
        ("n_times", C.c_int32),
        ("zero_mask", C.c_uint64),
        ("lo_mu", C.c_float),
        ("hi_mu", C.c_float),
        ("lo_sd", C.c_float),
        ("hi_sd", C.c_float),
    ]


class TrainHParams(C.Structure):
    """bnn_train_hparams (include/bnnchaos.h)."""

    _fields_ = [
        ("lr", C.c_float),
        ("momentum", C.c_float),
        ("weight_decay", C.c_float),
        ("clip_norm", C.c_float),
        ("beta_in", C.c_float),
        ("beta_out", C.c_float),
        ("first_step", C.c_int32),
        ("apply_update", C.c_int32),
    ]


class AdamHParams(C.Structure):
    """bnn_adam_hparams (include/bnnchaos.h)."""

    _fields_ = [
        ("beta1", C.c_double),
        ("beta2", C.c_double),
        ("eps", C.c_double),
        ("step", C.c_int64),
    ]


_CFG = C.POINTER(ModelConfig)
_HP = C.POINTER(TrainHParams)
_ADAM = C.POINTER(AdamHParams)

# name -> (restype, argtypes); must list every symbol of include/bnnchaos.h
SIGNATURES = {
    "bnn_abi_version": (C.c_int, []),
    "bnn_last_error_string": (C.c_char_p, []),
    "bnn_param_count": (C.c_int64, [_CFG]),
    "bnn_packed_param_count": (C.c_int64, [_CFG]),
    "bnn_swag_sample": (
        C.c_int,
        [_CFG, c_f32p, c_f32p, c_f32p, C.c_int32, C.c_int32, c_i32p, C.c_int64, C.c_int64, C.c_int32, C.c_float,
         C.c_uint64, c_f32p, c_f32p, c_f32p, c_f32p, C.c_void_p],
    ),
    "bnn_pack_theta": (C.c_int, [_CFG, c_f32p, C.c_int64, c_f32p, C.c_void_p]),
    "bnn_predict_workspace_bytes": (C.c_size_t, [_CFG, C.c_int64, C.c_int64]),
    "bnn_predict_system_granule": (C.c_int32, [_CFG]),
    "bnn_predict": (
        C.c_int,
        [_CFG, c_f32p, C.c_int64, c_f32p, C.c_int64, c_f32p, c_f32p, C.c_uint64, C.c_int64, C.c_int64, C.c_int32,
         c_f32p, c_f32p, C.c_void_p, C.c_void_p],
    ),
    "bnn_predict_strided": (
        C.c_int,
        [_CFG, c_f32p, C.c_int64, c_f32p, C.c_int64, c_f32p, c_f32p, C.c_uint64, C.c_int64, C.c_int64, C.c_int64,
         C.c_int64, c_f32p, c_f32p, C.c_void_p, C.c_void_p],
    ),
    "bnn_add_input_noise": (C.c_int, [_CFG, c_f32p, c_f32p, c_f32p, C.c_int64, c_f32p, C.c_void_p]),
    "bnn_predict_instability": (C.c_int, [_CFG, c_f32p, C.c_int64, c_f32p, c_f32p, C.c_void_p]),
    "bnn_multiswag_host_scratch_bytes": (C.c_size_t, [_CFG, C.c_int64, C.c_int64]),
    "bnn_multiswag_predict_host": (
        C.c_int,
        [_CFG, c_f32p, C.c_int64, c_f32p, c_f32p, c_f32p, C.c_int32, C.c_int32, C.c_int32, C.c_float, C.c_uint64,
         c_f32p, C.c_void_p, C.c_void_p],
    ),
    "bnn_nll_fwd_bwd": (C.c_int, [c_f32p, c_f32p, C.c_int64, c_f32p, c_f32p, c_f32p, C.c_void_p]),
    "bnn_train_workspace_bytes": (C.c_size_t, [_CFG, C.c_int64, C.c_int32]),
    "bnn_train_step": (
        C.c_int,
        [_CFG, _HP, C.c_int32, c_f32p, c_f32p, c_f32p, c_f32p, c_i32p, C.c_int64, c_f32p, c_f32p, c_f32p, C.c_uint64,
         C.c_uint64, c_f32p, c_f32p, C.c_void_p, C.c_void_p],
    ),
    "bnn_train_step_adam": (
        C.c_int,
        [_CFG, _HP, _ADAM, C.c_int32, c_f32p, c_f32p, c_f32p, c_f32p, c_f32p, c_i32p, C.c_int64, c_f32p, c_f32p, c_f32p,
         C.c_uint64, C.c_uint64, c_f32p, c_f32p, C.c_void_p, C.c_void_p],
    ),
    # per-seed hyperparameters: hp / adam are host arrays [n_seeds] (TrainHParams * n, AdamHParams * n), then plan_seeds
    "bnn_train_workspace_bytes_seeds": (C.c_size_t, [_CFG, C.c_int64, C.c_int32, C.c_int32]),
    "bnn_train_step_seeds": (
        C.c_int,
        [_CFG, _HP, C.c_int32, C.c_int32, c_f32p, c_f32p, c_f32p, c_f32p, c_i32p, C.c_int64, c_f32p, c_f32p, c_f32p, C.c_uint64,
         C.c_uint64, c_f32p, c_f32p, C.c_void_p, C.c_void_p],
    ),
    "bnn_train_step_adam_seeds": (
        C.c_int,
        [_CFG, _HP, _ADAM, C.c_int32, C.c_int32, c_f32p, c_f32p, c_f32p, c_f32p, c_f32p, c_i32p, C.c_int64, c_f32p, c_f32p, c_f32p,
         C.c_uint64, C.c_uint64, c_f32p, c_f32p, C.c_void_p, C.c_void_p],
    ),
    # per-seed halt: the _seeds arguments, then d_halted_at [n_seeds] int64 before the stream
    "bnn_train_step_seeds_halt": (
        C.c_int,
        [_CFG, _HP, C.c_int32, C.c_int32, c_f32p, c_f32p, c_f32p, c_f32p, c_i32p, C.c_int64, c_f32p, c_f32p, c_f32p, C.c_uint64,
         C.c_uint64, c_f32p, c_f32p, C.c_void_p, C.c_void_p, C.c_void_p],
    ),
    "bnn_train_step_adam_seeds_halt": (
        C.c_int,
        [_CFG, _HP, _ADAM, C.c_int32, C.c_int32, c_f32p, c_f32p, c_f32p, c_f32p, c_f32p, c_i32p, C.c_int64, c_f32p, c_f32p, c_f32p,
         C.c_uint64, C.c_uint64, c_f32p, c_f32p, C.c_void_p, C.c_void_p, C.c_void_p],
    ),
    "bnn_train_noise": (
        C.c_int,
        [_CFG, C.c_int32, C.c_int64, C.c_uint64, C.c_uint64, c_f32p, c_f32p, c_f32p, C.c_void_p],
    ),
    "bnn_eval_loss": (
        C.c_int,
        [_CFG, c_f32p, c_f32p, C.c_int64, c_f32p, C.c_int64, c_f32p, C.c_uint64, c_f32p, c_f32p, C.c_void_p,
         C.c_void_p],
    ),
    "bnn_swag_collect": (
        C.c_int,
        [c_f32p, C.c_int64, C.c_int32, C.c_int32, c_f32p, c_f32p, c_f32p, c_i32p, c_i32p, C.c_int32, C.c_int32,
         C.c_void_p],
    ),
    "bnn_swag_collect_halt": (
        C.c_int,
        [c_f32p, C.c_int64, C.c_int32, C.c_int32, c_f32p, c_f32p, c_f32p, c_i32p, c_i32p, C.c_int32, C.c_int32,
         C.c_void_p, C.c_void_p],
    ),
    "bnn_pack_inputs": (C.c_int, [c_f32p, c_f32p, c_f32p, c_f32p, C.c_int64, C.c_int32, c_f32p, C.c_void_p]),
    "bnn_sample_instability": (
        C.c_int, [c_f32p, C.c_int64, C.c_int64, C.c_uint64, C.c_int64, C.c_float, C.c_int32, c_f32p, C.c_void_p]),
    "bnn_summarize_instability": (C.c_int, [c_f32p, c_f32p, C.c_int64, C.c_int32, C.c_int32, c_f32p, C.c_void_p]),
    "bnn_score_labels": (C.c_int, [c_f32p, C.c_int64, C.c_int64, c_f32p, c_f32p, C.c_void_p]),
    "bnn_survival_instability": (
        C.c_int, [c_f32p, C.c_int64, C.c_int32, C.c_int64, C.POINTER(C.c_float), C.c_int32, c_f32p, C.c_void_p]),
    "bnn_summarize_instability_ragged": (
        C.c_int, [c_f32p, c_f32p, C.c_int64, C.c_void_p, C.c_int32, c_f32p, C.c_void_p]),
    "bnn_survival_instability_ragged": (
        C.c_int, [c_f32p, C.c_int64, C.c_void_p, C.c_int64, C.POINTER(C.c_float), C.c_int32, c_f32p, C.c_void_p]),
    "bnn_first_trio_instability": (C.c_int, [c_f32p, C.c_int64, C.c_int32, C.c_int64, c_f32p, C.c_void_p]),
    "bnn_first_trio_instability_ragged": (C.c_int, [c_f32p, C.c_int64, C.c_void_p, C.c_int64, c_f32p, C.c_void_p]),
    "bnn_decompose_uncertainty": (C.c_int, [c_f32p, C.c_int64, C.c_int64, C.c_int64, c_f32p, C.c_void_p]),
    "bnn_saliency": (C.c_int, [_CFG, C.c_int32, c_f32p, c_f32p, C.c_int64, c_f32p, C.c_uint64, c_f32p, c_f32p, c_f32p,
                               C.c_void_p, C.c_void_p]),
    "bnn_posterior_saliency_workspace_bytes": (C.c_size_t, [_CFG, C.c_int32, C.c_int64]),
    "bnn_posterior_saliency": (
        C.c_int,
        [_CFG, C.c_int32, c_f32p, C.c_int64, c_f32p, C.c_int64, C.c_int64, C.c_uint64, C.c_void_p, C.c_int32, C.c_int64,
         c_f32p, c_f32p, c_f32p, C.c_void_p, C.c_void_p],
    ),
    "bnn_integrate_orbits": (
        C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_double, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
}

# diagnostics declared in include/bnnchaos_diag.h (probes / timers; not part of the product ABI)
DIAG_SIGNATURES = {
    "bnn_ffma_peak": (C.c_int, [C.c_int32, C.c_int64, c_f32p, C.POINTER(C.c_int64), C.c_void_p]),
    "bnn_tc_probe": (C.c_int, [c_f32p, c_f32p, c_f32p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "bnn_tc_time": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]),
    "bnn_train_timeline": (C.c_int, [C.POINTER(C.c_ulonglong), C.c_int32]),
    "bnn_mma_sync_rate": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_void_p, c_f32p, C.c_void_p]),
    "bnn_swag_sample_unfused": (
        C.c_int,
        [_CFG, c_f32p, c_f32p, c_f32p, C.c_int32, C.c_int32, c_i32p, C.c_int64, C.c_int64, C.c_int32, C.c_float,
         C.c_uint64, c_f32p, c_f32p, c_f32p, c_f32p, C.c_void_p],
    ),
    "bnn_set_train_variant": (C.c_int, [C.c_int32]),
    "bnn_set_train_seed_groups": (C.c_int, [C.c_int32]),
    "bnn_train_seed_plan": (C.c_int, [_CFG, C.c_int64, C.c_int32, c_i32p, c_i32p, c_i32p]),
    "bnn_set_summary_variant": (C.c_int, [C.c_int32]),
    "bnn_set_predict_variant": (C.c_int, [C.c_int32]),
    "bnn_set_predict_unit_chunk": (C.c_int, [C.c_int64]),
    "bnn_tc_probe_ss": (C.c_int, [c_f32p, c_f32p, c_f32p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                  C.c_int32, C.c_void_p]),
}

_lib = None


class BnnChaosError(RuntimeError):
    pass


def load():
    """Load libbnnchaos.so once; raise ImportError loudly when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build the CUDA extension first "
            "(python -c 'import __graft_entry__ as g; g.build()' or make -C bnn_chaos_model_b200/csrc). "
            "This package has no CPU fallback."
        )
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in list(SIGNATURES.items()) + list(DIAG_SIGNATURES.items()):
        fn = getattr(lib, name)  # AttributeError if the library does not export it
        fn.restype = res
        fn.argtypes = args
    if lib.bnn_abi_version() != 1:
        raise ImportError(f"libbnnchaos ABI version {lib.bnn_abi_version()} != 1; rebuild the extension")
    _lib = lib
    return lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = load().bnn_last_error_string().decode("utf-8", "replace")
        kind = "CUDA error" if rc > 0 else "argument error"
        raise BnnChaosError(f"{what or 'libbnnchaos'}: {kind} {rc}: {msg}")


def ptr(t):
    """Device/host pointer of a contiguous tensor (or None)."""
    if t is None:
        return None
    assert t.is_contiguous(), "libbnnchaos needs contiguous tensors"
    return t.data_ptr()


def dev_ptr(t, device, name, dtype=None):
    """Pointer of a tensor the kernels will dereference ON `device`: raises BnnChaosError unless the tensor lives on
    exactly that device, is contiguous and has the expected dtype (default float32) -- a tensor on another GPU would
    otherwise be read through a foreign address, a float64 / int64 tensor as fp32 words."""
    import torch

    if t is None:
        return None
    dtype = torch.float32 if dtype is None else dtype
    device = torch.device(device)
    if not t.is_cuda:
        require_cuda(t, name)
    if device.index is None:
        device = torch.device("cuda", torch.cuda.current_device())
    if t.device != device:
        raise BnnChaosError(f"{name} is on {t.device} but the launch device is {device}: move it first")
    if t.dtype != dtype:
        raise BnnChaosError(f"{name} has dtype {t.dtype}; the kernels read {dtype}")
    if not t.is_contiguous():
        raise BnnChaosError(f"{name} must be contiguous")
    return t.data_ptr()


class nvtx:
    """NVTX range around a launch group (K1 sample / K2 predict / K4 train step / K6 pack / K7 posterior), visible in
    nsys / ncu timelines (SURVEY.md section 5).  A no-op costing two host calls when no profiler is attached."""

    def __init__(self, name):
        self.name = name

    def __enter__(self):
        import torch

        torch.cuda.nvtx.range_push(self.name)
        return self

    def __exit__(self, *exc):
        import torch

        torch.cuda.nvtx.range_pop()
        return False


def current_stream_ptr():
    import torch

    return torch.cuda.current_stream().cuda_stream


def require_cuda(t, name):
    if not t.is_cuda:
        raise BnnChaosError(
            f"{name} is on {t.device}: the B200 path has no CPU fallback; move it to a CUDA device "
            "(the CPU restatement lives in oracle/ and is test infrastructure only)"
        )
