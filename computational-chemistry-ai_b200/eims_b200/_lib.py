"""ctypes binding of libeims_b200.so (the C ABI declared in include/eims_b200.h).

There is deliberately no fallback: if the CUDA library is missing or the device is not a
B200-class (sm_100) GPU, importing / using this module raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# EIMS_LIB: another build of the same library (A/B timing of kernel variants); never a different implementation
LIB_PATH = os.environ.get("EIMS_LIB") or os.path.join(_HERE, "libeims_b200.so")

POOLING = {"sum": 0, "mean": 1, "max": 2, "combined": 3}
LOSS = {"mse": 0, "cosine": 1}
GEMM_TCGEN05, GEMM_FP32_SIMT = 0, 1
BWD_ALL, BWD_HEAD, BWD_GCN = 0, 1, 2

ERR_ARG, ERR_CUDA, ERR_CAPACITY, ERR_ZERO_DEGREE, ERR_STATE = -1, -2, -3, -4, -5


class EimsError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"eims_b200 error {code}: {msg}")
        self.code = code


class ZeroInDegreeError(EimsError):
    """Mirrors DGLError('There are 0-in-degree nodes in the graph ...') raised by GraphConv."""


class Dims(C.Structure):
    _fields_ = [("node_feat_dim", C.c_int32), ("hidden_dim", C.c_int32), ("num_gcn_layers", C.c_int32),
                ("max_mz", C.c_int32), ("pooling", C.c_int32), ("dropout", C.c_float)]


class Peaks(C.Structure):
    _fields_ = [("peak_ptr", C.c_void_p), ("mz", C.c_void_p), ("intensity", C.c_void_p),
                ("mz_is_f64", C.c_int32), ("num_spectra", C.c_int64)]


class Dataset(C.Structure):
    _fields_ = [("node_ptr", C.c_void_p), ("bond_ptr", C.c_void_p), ("feat", C.c_void_p),
                ("bond_begin", C.c_void_p), ("bond_end", C.c_void_p), ("targets", C.c_void_p),
                ("num_mols", C.c_int64), ("peaks", C.POINTER(Peaks))]


class HostBatchLayout(C.Structure):
    _fields_ = [(n, C.c_int64) for n in ("node_ptr", "bond_ptr", "bond_begin", "bond_end", "feat", "targets", "peak_ptr",
                                         "peak_mz", "peak_inten", "nbytes")] + \
               [(n, C.c_int32) for n in ("num_graphs", "num_nodes", "num_edges", "feat_dim", "mz_is_f64")]


class GemmProblem(C.Structure):
    """eims_gemm_problem: one product of eims_gemm_planes."""
    _fields_ = [("A", C.c_void_p), ("lda", C.c_int32), ("a_mn_major", C.c_int32),
                ("B", C.c_void_p), ("ldb", C.c_int32), ("b_mn_major", C.c_int32),
                ("C", C.c_void_p), ("ldc", C.c_int32),
                ("M", C.c_int32), ("N", C.c_int32), ("K", C.c_int32),
                ("m_dev", C.c_void_p), ("k_dev", C.c_void_p), ("row_scale", C.c_void_p), ("bias", C.c_void_p),
                ("relu", C.c_int32), ("accumulate", C.c_int32)]


class Step(C.Structure):
    _fields_ = [("lr", C.c_float), ("beta1", C.c_float), ("beta2", C.c_float), ("eps", C.c_float),
                ("weight_decay", C.c_float), ("grad_scale", C.c_float), ("step", C.c_int32), ("seed", C.c_uint64)]


_vp, _i32, _i64, _f32, _u64 = C.c_void_p, C.c_int32, C.c_int64, C.c_float, C.c_uint64
_SIGS = {
    "eims_version": (C.c_int, []),
    "eims_last_error": (C.c_char_p, []),
    "eims_device_check": (C.c_int, []),
    "eims_param_count": (_i64, [C.POINTER(Dims)]),
    "eims_param_num_tensors": (C.c_int, [C.POINTER(Dims)]),
    "eims_param_layout": (C.c_int, [C.POINTER(Dims), C.POINTER(_i64), _i32]),
    "eims_peaks_to_spectrum": (C.c_int, [C.POINTER(Peaks), _vp, _i32, _i32, _vp, _vp]),
    "eims_topk_peaks": (C.c_int, [_vp, _i32, _i32, _i32, _vp, _vp, _vp]),
    "eims_plan_set_peak_targets": (C.c_int, [_vp, C.POINTER(Peaks)]),
    "eims_csr_build": (C.c_int, [C.POINTER(Dataset), _vp, _i32, _i32, _i32, _i32] + [_vp] * 10 + [_vp]),
    "eims_spmm_norm": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i32, _vp, _vp, _f32, _u64, _i32, _i32, _i32, _vp, _i32, _vp]),
    "eims_spmm_norm_mol": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _i32, _vp, _vp, _f32, _u64, _i32, _i32, _i32, _vp, _i32, _i32, _i32, _vp]),
    "eims_gemm": (C.c_int, [_i32, _vp, _i32, _i32, _vp, _i32, _i32, _vp, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _i32, _i32, _vp]),
    "eims_gemm_planes_scratch_bytes": (_i64, [C.POINTER(GemmProblem), C.POINTER(GemmProblem)]),
    "eims_gemm_planes": (C.c_int, [C.POINTER(GemmProblem), C.POINTER(GemmProblem), _vp, _i64, _vp]),
    "eims_bn_scratch_floats": (_i64, [_i32, _i32]),
    "eims_bn_stats": (C.c_int, [_vp, _vp, _i32] + [_vp] * 9 + [_i32, _vp]),
    "eims_readout": (C.c_int, [_vp, _vp, _vp, _i32, _vp, _vp, _i32, _vp, _vp, _i32, _vp]),
    "eims_loss_mse_cos": (C.c_int, [_vp, _vp, _vp, _vp, _i32, _i32, _vp, _vp, _vp, _vp, _i32, _vp]),
    "eims_adamw_flat": (C.c_int, [_vp, _vp, _vp, _vp, _i64, C.POINTER(Step), _vp]),
    "eims_dropout_mask": (C.c_int, [_f32, _u64, _i32, _i32, _i32, _i32, _vp, _vp]),
    "eims_plan_create": (C.c_int, [C.POINTER(Dims), _i32, _i32, _i32, C.POINTER(_vp)]),
    "eims_plan_destroy": (C.c_int, [_vp]),
    "eims_plan_workspace_bytes": (_i64, [_vp]),
    "eims_plan_bind": (C.c_int, [_vp, _vp, _i64]),
    "eims_plan_set_gemm_backend": (C.c_int, [_vp, _i32]),
    "eims_plan_set_gemm_planes": (C.c_int, [_vp, _i32]),
    "eims_plan_buffer": (C.c_int, [_vp, C.c_char_p, C.POINTER(_vp), C.POINTER(_i64)]),
    "eims_batch_build": (C.c_int, [_vp, C.POINTER(Dataset), _vp, _i32, _vp]),
    "eims_forward": (C.c_int, [_vp, _vp, _vp, _i32, C.POINTER(Step), _vp]),
    "eims_sigmoid": (C.c_int, [_vp, _vp]),
    "eims_loss": (C.c_int, [_vp, _vp, _vp, _i32, _i32, _vp]),
    "eims_backward": (C.c_int, [_vp, _vp, _vp, _vp, _vp]),
    "eims_backward_part": (C.c_int, [_vp, _vp, _vp, _vp, _i32, _vp]),
    "eims_backward_feat": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "eims_attribute_peaks": (C.c_int, [_vp, _vp, _vp, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp]),
    "eims_metrics_accumulate": (C.c_int, [_vp, _vp, _vp]),
    "eims_train_step": (C.c_int, [_vp, C.POINTER(Dataset), _vp, _i32, _vp, _vp, _vp, _vp, _vp, _i32, C.POINTER(Step), _vp, _vp]),
    "eims_train_step_built": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, C.POINTER(Step), _vp, _vp]),
    "eims_infer_batch": (C.c_int, [_vp, C.POINTER(Dataset), _vp, _i32, _vp, _vp, _vp, _vp]),
    "eims_dp_adamw_fused": (C.c_int, [_i32, _i32, C.POINTER(_u64), C.POINTER(_u64), C.POINTER(_u64), _u64, _u64, _vp, _vp, _vp,
                                      _i64, _i64, C.POINTER(Step), C.c_uint32, _i32, _vp, _vp]),
    "eims_dp_adamw_fused_blk": (C.c_int, [_i32, _i32, C.POINTER(_u64), C.POINTER(_u64), C.POINTER(_u64), _u64, _u64, _vp, _vp, _vp,
                                          _i64, _i64, C.POINTER(Step), C.c_uint32, _i32, _vp, _vp, _vp]),
    "eims_host_pack_batch": (C.c_int, [C.POINTER(Dataset), _vp, _i32, _i32, _i32, _vp, _i64, C.POINTER(HostBatchLayout)]),
    "eims_host_pack_batch_fixed": (C.c_int, [C.POINTER(Dataset), _vp, _i32, _i32, _i32, _i64, _i64, _i64, _vp, _i64, C.POINTER(HostBatchLayout)]),
    "eims_step_block_bytes": (_i64, []),
    "eims_plan_set_step_block": (C.c_int, [_vp, _vp, _i64]),
    "eims_step_block_upload": (C.c_int, [_vp, C.POINTER(Step), _vp, C.c_uint32, _vp]),
    "eims_plan_select_step_block": (C.c_int, [_vp, _i32]),
    "eims_step_blocks_upload": (C.c_int, [_vp, C.POINTER(Step), C.POINTER(_vp), C.POINTER(C.c_uint32), _i32, _i32, _vp]),
    "eims_batch_build_indirect": (C.c_int, [_vp, C.POINTER(Dataset), _i32, _vp]),
    "eims_train_step_built_indirect": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _vp, _vp, _vp]),
    "eims_train_step_built_indirect_part": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i32, _vp, _i32, _vp]),
    "eims_plan_profile": (C.c_int, [_vp, _i32]),
    "eims_plan_profile_read": (C.c_int, [_vp, C.POINTER(_f32), C.POINTER(_i32), _i32, C.POINTER(_i64)]),
    "eims_plan_num_stages": (C.c_int, []),
    "eims_plan_stage_name": (C.c_char_p, [_i32]),
    "eims_plan_check": (C.c_int, [_vp, C.POINTER(_i32), C.POINTER(_i32), _vp]),
}

EXPORTS = tuple(_SIGS)
_lib = None


def load() -> C.CDLL:
    """Load the shared library (no device needed for this; compute calls need a B200)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing. Build it with `python computational-chemistry-ai_b200/build.py` "
                "(nvcc, sm_100a). There is no CPU or other-GPU fallback.")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
        _lib = lib
    return _lib


def check(rc: int) -> None:
    if rc == 0:
        return
    msg = load().eims_last_error().decode(errors="replace")
    if rc == ERR_ZERO_DEGREE:
        raise ZeroInDegreeError(rc, msg)
    raise EimsError(rc, msg)


def ptr(t):
    """Device / host pointer of a torch tensor or an address (None -> NULL)."""
    return None if t is None else C.c_void_p(t if isinstance(t, int) else t.data_ptr())
