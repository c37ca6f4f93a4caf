"""ctypes binding of libdagma_b200.so (the C ABI declared in include/dagma_b200.h).

There is no fallback: if the shared library is missing or the device is not a
compute-capability-10.x GPU, every entry point raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# DAGMA_B200_LIB: another build of the same sources (A/B timing and debug builds, scripts/build_variant.py)
LIB_PATH = os.environ.get("DAGMA_B200_LIB") or os.path.join(_HERE, "lib", "libdagma_b200.so")

MAX_STAGES = 16
SMALL_MAX_D = 64
ONCHIP_INV_MAX_D = 128
DIAG_COLS = 11

ST_OK, ST_OUT_OF_DOMAIN, ST_LR_UNDERFLOW, ST_RETRY_LIMIT = 0, 1, 2, 4
ST_PERRON_CAP = 8                # TCC batches: some Perron solve hit the chunk cap


class SmallFitArgs(C.Structure):
    """mirror of ``dagma_small_fit_args`` (include/dagma_b200.h)"""
    _fields_ = [
        ("batch", C.c_int32), ("d", C.c_int32), ("n_stages", C.c_int32), ("checkpoint", C.c_int32),
        ("retry_on_fail", C.c_int32), ("ckpt_log_cap", C.c_int32),
        ("lr", C.c_double), ("tol", C.c_double), ("beta1", C.c_double), ("beta2", C.c_double),
        ("mu", C.c_double * MAX_STAGES), ("s", C.c_double * MAX_STAGES), ("iters", C.c_int32 * MAX_STAGES),
        ("cov", C.c_void_p), ("lambda1", C.c_void_p), ("w", C.c_void_p),
        ("mask_exc", C.c_void_p), ("mask_inc", C.c_void_p),
        ("status", C.c_void_p), ("stage_stats", C.c_void_p), ("final", C.c_void_p),
        ("ckpt_log", C.c_void_p), ("ckpt_count", C.c_void_p), ("work_counter", C.c_void_p),
        ("ckpt_diag", C.c_void_p),
    ]


EXPORTS = {
    # name: (restype, argtypes)
    "dagma_version": (C.c_int, []),
    "dagma_last_error": (C.c_char_p, []),
    "dagma_device_check": (C.c_int, [C.POINTER(C.c_int)]),
    "dagma_logdet_inv_f64": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_void_p, C.c_int, C.c_int,
                                       C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                       C.c_void_p, C.c_void_p]),
    "dagma_linear_fit_small_f64": (C.c_int, [C.c_void_p, C.POINTER(SmallFitArgs)]),
    "dagma_linear_fit_small_logistic_f64": (C.c_int, [C.c_void_p, C.POINTER(SmallFitArgs), C.c_int, C.c_void_p]),
    "dagma_linear_fit_small_pst_f64": (C.c_int, [C.c_void_p, C.POINTER(SmallFitArgs), C.c_void_p, C.c_void_p,
                                                 C.c_void_p, C.c_int, C.c_double]),
    "dagma_linear_fit_small_pst_exp_f64": (C.c_int, [C.c_void_p, C.POINTER(SmallFitArgs), C.c_void_p, C.c_void_p,
                                                     C.c_void_p, C.c_int]),
    "dagma_linear_fit_small_tcc_f64": (C.c_int, [C.c_void_p, C.POINTER(SmallFitArgs), C.c_void_p, C.c_void_p,
                                                 C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                                 C.c_void_p]),
    "dagma_linear_fit_small_geometry": (C.c_int, [C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int),
                                                  C.POINTER(C.c_size_t)]),
    "dagma_fit_dmma_residency": (C.c_int, [C.POINTER(C.c_int)]),
    "dagma_linear_fit_small_host_f64": (C.c_int, [C.c_void_p, C.POINTER(SmallFitArgs)]),
    "dagma_gemm_f64": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, C.c_void_p, C.c_int,
                                 C.c_void_p, C.c_int, C.c_double, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_size_t]),
    "dagma_large_workspace_bytes": (C.c_size_t, [C.c_int]),
    "dagma_logdet_inv_ws_f64": (C.c_int, [C.c_void_p, C.c_int, C.c_double, C.c_void_p, C.c_int, C.c_int,
                                          C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                          C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "dagma_logdet_inv_gemm_ws_f64": (C.c_int, [C.c_void_p, C.c_int, C.c_double, C.c_void_p, C.c_int, C.c_int,
                                               C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                               C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t,
                                               C.c_void_p, C.c_void_p, C.c_void_p]),
    "dagma_linear_update_f64": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                          C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "dagma_linear_update_ex_f64": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                             C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                             C.c_double]),
    "dagma_linear_apply_dir_f64": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                             C.c_double]),
    "dagma_linear_iter_supported": (C.c_int, [C.c_int, C.c_int, C.c_int]),
    "dagma_linear_iter_workspace_doubles": (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    "dagma_linear_iter_f64": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "dagma_linear_iter_exchange_bytes": (C.c_size_t, [C.c_int, C.c_int]),
    "dagma_linear_iter_sharded_f64": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                                C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                                C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "dagma_graph_metrics": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "dagma_peer_alloc": (C.c_int, [C.c_size_t, C.c_void_p]),
    "dagma_peer_free": (C.c_int, [C.c_void_p]),
    "dagma_peer_export": (C.c_int, [C.c_void_p, C.c_void_p]),
    "dagma_peer_import": (C.c_int, [C.c_void_p, C.c_void_p]),
    "dagma_peer_release": (C.c_int, [C.c_void_p]),
    "dagma_stream_create": (C.c_int, [C.c_void_p]),
    "dagma_stream_destroy": (C.c_int, [C.c_void_p]),
    "dagma_linear_objective_f64": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                             C.c_int]),
    "dagma_linear_objective_workspace_bytes": (C.c_size_t, []),
    "dagma_linear_objective_ws_f64": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                                C.c_int, C.c_void_p, C.c_size_t]),
    "dagma_logistic_loss_f64": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_double,
                                          C.c_void_p, C.c_int, C.c_void_p]),
    "dagma_adam_direction_f64": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_double,
                                           C.c_double, C.c_double, C.c_double, C.c_void_p]),
    "dagma_mlp_adj_f64": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "dagma_mlp_forward_f64": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "dagma_mlp_objective_f64": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int]),
    "dagma_mlp_backward_f64": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.c_void_p, C.c_void_p]),
    "dagma_mlp_adam_f64": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_void_p]),
    "dagma_mlp_adam_ex_f64": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_void_p, C.c_void_p]),
    "dagma_mlp_iter_supported": (C.c_int, [C.c_int, C.c_int, C.c_int]),
    "dagma_mlp_iter_workspace_doubles": (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    "dagma_mlp_iter_f64": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "dagma_mlp_iter_exchange_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    "dagma_mlp_iter_sharded_f64": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                             C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                             C.c_int, C.c_int, C.c_void_p]),
    "dagma_mlp_batch_supported": (C.c_int, [C.c_int, C.c_int, C.c_int]),
    "dagma_mlp_minimize_batch_f64": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                               C.c_double, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                               C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "dagma_lc_forward_f64":(C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_void_p]),
    "dagma_mlp_residual_f64": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "dagma_lc_backward_f64": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_void_p]),
    "dagma_row_sums_f64": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "dagma_locally_connected_f64": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                              C.c_void_p, C.c_void_p]),
    "dagma_sumsq_diff_f64": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "dagma_tcc_assemble_f64": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_double, C.c_int, C.c_void_p]),
    "dagma_power_workspace_bytes": (C.c_size_t, [C.c_int]),
    "dagma_perron_power_f64": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_int,
                                         C.c_double, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.c_size_t]),
    "dagma_matvec_f64": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "dagma_vec_dots_f64": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "dagma_rank2_fold_f64": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_double, C.c_void_p, C.c_double, C.c_int, C.c_void_p]),
    "dagma_tcc_fold_f64": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_double, C.c_int, C.c_void_p]),
    "dagma_center_cov_f64": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p]),
    "dagma_mi_upper_d2_f64": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "dagma_mi_centered_gram_f64": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                             C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "dagma_mi_perm_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    "dagma_mi_perm_dots_f64": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.c_int, C.c_double, C.c_void_p, C.c_size_t, C.c_void_p]),
    "dagma_bench_fp64_fma": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "dagma_bench_fp64_dmma": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "dagma_bench_latency": (C.c_int, [C.c_void_p, C.c_void_p]),
    "dagma_bench_stage": (C.c_int, [C.c_void_p, C.c_void_p]),
    "dagma_bench_engine_gemm": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "dagma_bench_tma_gemm": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int,
                                       C.c_void_p, C.c_int, C.c_double, C.c_double, C.c_int, C.c_void_p]),
    "dagma_bench_fp64_dmma_tiles": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
}

_lib = None


class DagmaB200Error(RuntimeError):
    pass


def load() -> C.CDLL:
    """dlopen the library once and bind every exported symbol."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise DagmaB200Error(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). midagma_b200 has no CPU or PyTorch fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in EXPORTS.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is missing
        fn.restype, fn.argtypes = res, args
    _lib = lib
    return lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load().dagma_last_error().decode(errors="replace")
        raise DagmaB200Error(f"{what or 'libdagma_b200'} failed (rc={rc}): {msg}")


_device_ok = {}


def require_device() -> int:
    """Fail loudly unless the current CUDA device is a B200-class (sm_100) GPU."""
    import torch
    if not torch.cuda.is_available():
        raise DagmaB200Error("midagma_b200 needs a CUDA device (sm_100a); there is no CPU path")
    dev = torch.cuda.current_device()
    if dev not in _device_ok:
        torch.cuda.init()
        sms = C.c_int(0)
        check(load().dagma_device_check(C.byref(sms)), "dagma_device_check")
        _device_ok[dev] = sms.value
    return _device_ok[dev]


def stream_ptr() -> int:
    import torch
    return torch.cuda.current_stream().cuda_stream
