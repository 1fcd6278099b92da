"""ctypes binding of libicpcuda.so (include/icpcuda.h). Fails loudly when the CUDA library is missing:
there is no CPU fallback anywhere in this package."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# ICPCUDA_LIB_TAG selects an experiment build of the same CUDA library (tools/fused_timing.py); default: the product build
LIB_PATH = os.path.join(_HERE, "libicpcuda" + ("_" + os.environ["ICPCUDA_LIB_TAG"] if os.environ.get("ICPCUDA_LIB_TAG") else "") + ".so")

OK = 0
ERR_INVALID_ARGUMENT, ERR_CUDA, ERR_OUT_OF_MEMORY, ERR_EMPTY_SET, ERR_NOT_POSITIVE_DEFINITE, ERR_NAN = -1, -2, -3, -4, -5, -6
CHAIN_EMPTY_SET, CHAIN_NOT_POSITIVE_DEFINITE, CHAIN_NAN_TRANSITION, CHAIN_NAN_VALUE = 1, 2, 4, 8
FACTOR_CHOLESKY, FACTOR_SVD = 0, 1
RANK_UPDATE_FP64, RANK_UPDATE_INT8 = 0, 1
MODEL_SAMPLING, TARGET_SAMPLING, MODEL_AND_TARGET_SAMPLING = 0, 1, 2
STD_ICP_NON_FINITE, STD_ICP_NOT_POSITIVE_DEFINITE = 1, 2
EVAL_ACCEPT_ALL, EVAL_INDEPENDENT, EVAL_HAUSDORFF, EVAL_COLLECTIVE = 0, 1, 2, 3
MODEL_TO_TARGET, TARGET_TO_MODEL, SYMMETRIC = 0, 1, 2
PROP_ICP, PROP_RANDOM_SHAPE, PROP_ROTATION, PROP_TRANSLATION = 0, 1, 2, 3
N_STAGES = 11

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int32)
_bp = C.POINTER(C.c_uint8)
_lp = C.POINTER(C.c_int64)
_h = C.c_void_p


class IcpCudaError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libicpcuda error {code}: {msg}")
        self.code = code


class ProposalParams(C.Structure):
    _fields_ = [("step_length", C.c_double), ("tangential_noise", C.c_double), ("noise_along_normal", C.c_double),
                ("direction", C.c_int32), ("boundary_aware", C.c_int32), ("factor", C.c_int32), ("rank_update", C.c_int32)]


class EvaluatorParams(C.Structure):
    _fields_ = [("kind", C.c_int32), ("mode", C.c_int32), ("use_prior", C.c_int32), ("reserved", C.c_int32),
                ("p0", C.c_double), ("p1", C.c_double), ("p2", C.c_double)]


class Component(C.Structure):
    _fields_ = [("kind", C.c_int32), ("axis", C.c_int32), ("weight", C.c_double), ("sd", C.c_double), ("proposal", _h)]


class ChainTarget(C.Structure):
    _fields_ = [("target", _h), ("components", C.POINTER(Component)), ("evaluator", _h)]


class KernelTerm(C.Structure):
    _fields_ = [("scale", C.c_double), ("sigma", C.c_double), ("A", C.c_double * 9)]


class FaceKernel(C.Structure):
    _fields_ = [("n_levels", C.c_int32), ("level", C.c_int32 * 8), ("scale", C.c_double * 8), ("symmetric_weight", C.c_double),
                ("plain_weight", C.c_double)]


class ChainIO(C.Structure):
    _fields_ = [("seed", C.c_uint64), ("chain_id_offset", C.c_uint64), ("u_comp", C.c_void_p), ("z", C.c_void_p),
                ("u_acc", C.c_void_p), ("log_component", C.c_void_p), ("log_accepted", C.c_void_p),
                ("log_values", C.c_void_p), ("log_theta", C.c_void_p), ("theta_final", C.c_void_p),
                ("n_accepted", C.c_void_p), ("status", C.c_void_p), ("theta_best", C.c_void_p), ("value_best", C.c_void_p),
                ("metrics_interval", C.c_int32), ("reserved", C.c_int32), ("log_metrics", C.c_void_p)]


class StdIcpIO(C.Structure):
    _fields_ = [("seed", C.c_uint64), ("fit_id_offset", C.c_uint64), ("directions", C.c_void_p), ("alpha_final", C.c_void_p),
                ("log_alpha", C.c_void_p), ("log_direction", C.c_void_p), ("status", C.c_void_p), ("iterations_done", C.c_void_p)]


class StdIcpTarget(C.Structure):
    _fields_ = [("target", _h), ("target_points", _dp)]


class ChainStatsParams(C.Structure):
    _fields_ = [("burn_in", C.c_int64), ("take_every_n", C.c_int64), ("end", C.c_int64), ("normals", C.c_int32),
                ("reserved", C.c_int32)]


_SIGS = {
    "icp_ctx_create": [C.c_int32, C.POINTER(_h)],
    "icp_ctx_destroy": [_h],
    "icp_last_error": [_h, C.c_char_p, C.c_size_t],
    "icp_version": [_h, C.c_char_p, C.c_size_t],
    "icp_model_create": [_h, C.c_int32, C.c_int32, C.c_int32, _dp, _dp, _dp, _dp, _ip, C.POINTER(_h)],
    "icp_model_destroy": [_h],
    "icp_model_rank": [_h, _ip],
    "icp_target_create": [_h, C.c_int32, C.c_int32, _dp, _ip, C.POINTER(_h)],
    "icp_target_destroy": [_h],
    "icp_closest_point_surface": [_h, C.c_int64, _dp, _ip, _ip, _dp, _dp],
    "icp_closest_point_surface_device": [_h, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p],
    "icp_closest_vertex": [_h, C.c_int64, _dp, _ip, _dp],
    "icp_target_boundary_flags": [_h, _bp],
    "icp_reconstruct": [_h, C.c_int32, _dp, _dp],
    "icp_vertex_normals": [_h, C.c_int32, _dp, _dp],
    "icp_model_closest_point_surface": [_h, C.c_int32, _dp, C.c_int64, _dp, _ip, _ip, _dp, _dp],
    "icp_model_closest_vertex": [_h, C.c_int32, _dp, C.c_int64, _dp, _ip, _dp],
    "icp_model_boundary_flags": [_h, _bp],
    "icp_proposal_create": [_h, _h, C.POINTER(ProposalParams), _ip, C.c_int32, _dp, C.c_int32, C.POINTER(_h)],
    "icp_proposal_destroy": [_h],
    "icp_posterior": [_h, C.c_int32, _dp, _dp, _dp, _ip],
    "icp_propose": [_h, C.c_int32, _dp, _dp, _dp],
    "icp_log_transition": [_h, C.c_int32, _dp, _dp, _dp],
    "icp_proposal_clear_cache": [_h],
    "icp_std_icp_iteration": [_h, _h, C.c_int32, _ip, C.c_int32, _dp, C.c_int32, C.c_double, C.c_double, C.c_int32, _dp, _dp],
    "icp_std_icp_iteration_theta": [_h, _h, C.c_int32, _ip, C.c_int32, _dp, C.c_int32, C.c_double, C.c_double, C.c_int32, _dp, _dp],
    "icp_std_icp_create": [_h, _h, _ip, C.c_int32, _dp, C.c_int32, C.c_double, C.c_int32, C.c_int32, C.POINTER(_h)],
    "icp_std_icp_create_targets": [_h, C.c_int32, C.POINTER(StdIcpTarget), _ip, C.c_int32, C.c_int32, C.c_double, C.c_int32,
                                   C.c_int32, C.POINTER(_h)],
    "icp_std_icp_set_target_index": [_h, C.c_int32, _ip],
    "icp_std_icp_destroy": [_h],
    "icp_std_icp_run": [_h, C.c_int32, _dp, C.c_int32, _dp, C.c_int32, C.POINTER(StdIcpIO)],
    "icp_std_icp_run_device": [_h, C.c_int32, C.c_void_p, C.c_int32, _dp, C.c_int32, C.POINTER(StdIcpIO), C.c_int32],
    "icp_std_icp_last_run_stats": [_h, _dp, _lp],
    "icp_evaluator_create": [_h, _h, C.POINTER(EvaluatorParams), _ip, C.c_int32, _dp, C.c_int32, C.POINTER(_h)],
    "icp_evaluator_destroy": [_h],
    "icp_eval_log_value": [_h, C.c_int32, _dp, _dp, _ip],
    "icp_eval_prior": [_h, C.c_int32, _dp, _dp],
    "icp_registration_metrics": [_h, _h, C.c_int32, _dp, _dp],
    "icp_dice_coefficient": [_h, _h, C.c_int32, _dp, C.c_int32, _dp, C.c_uint64, _dp],
    "icp_registration_metrics_targets": [_h, C.c_int32, C.POINTER(_h), C.c_int32, _dp, _ip, _dp],
    "icp_dice_coefficient_targets": [_h, C.c_int32, C.POINTER(_h), C.c_int32, _dp, _ip, C.c_int32, _dp, C.c_uint64, _dp],
    "icp_posterior_variability": [_h, C.c_int32, _dp, C.c_int32, _dp, _dp, _dp, _dp, _dp],
    "icp_gpmm_kernel_matrix": [_h, C.c_int32, _dp, C.c_int32, _dp, C.POINTER(KernelTerm), C.c_int32, _dp],
    "icp_gpmm_eigen_psd": [_h, C.c_int32, _dp, C.c_int32, _dp, _dp],
    "icp_gpmm_nystrom_extend": [_h, C.c_int32, _dp, C.c_int32, _dp, C.POINTER(KernelTerm), C.c_int32, C.c_int32, _dp, _dp, _dp, _dp],
    "icp_gpmm_face_kernel_matrix": [_h, C.c_int32, _dp, _dp, C.c_int32, _dp, _dp, _dp, C.POINTER(FaceKernel), _dp],
    "icp_gpmm_face_nystrom_extend": [_h, C.c_int32, _dp, _dp, C.c_int32, _dp, _dp, _dp, C.POINTER(FaceKernel), C.c_int32, _dp, _dp, _dp, _dp],
    "icp_jsonlog_open": [C.c_char_p, C.c_int32, C.POINTER(C.c_char_p), C.c_int32, C.POINTER(C.c_char_p), C.POINTER(_h)],
    "icp_jsonlog_append": [_h, C.c_int32, C.c_int32, C.c_int32, _ip, _bp, _dp, _dp],
    "icp_jsonlog_close": [_h],
    "icp_jsonlog_load": [C.c_char_p, C.c_int32, C.c_int64, _lp, _lp, _bp, _dp, _dp, C.c_char_p, C.c_char_p],
    "icp_chainlog_sample_indices": [C.c_int64, _bp, C.c_int32, C.c_int64, C.c_int64, C.c_int64, _lp, _lp],
    "icp_comm_unique_id": [_h, _bp],
    "icp_comm_init": [_h, C.c_int32, C.c_int32, _bp, C.POINTER(_h)],
    "icp_comm_destroy": [_h],
    "icp_comm_info": [_h, _ip, _ip, _ip],
    "icp_chainlog_gather": [_h, C.c_int32, C.c_int32, C.c_int32, C.POINTER(ChainIO), C.POINTER(ChainIO), _dp, _lp],
    "icp_variability_allreduce": [_h, _h, C.c_int32, _dp, C.c_int32, _dp, _dp, _dp, _dp, _dp, _lp],
    "icp_chain_create": [_h, _h, C.POINTER(Component), C.c_int32, _h, C.c_int32, C.POINTER(_h)],
    "icp_chain_create_targets": [_h, C.c_int32, C.POINTER(ChainTarget), C.c_int32, C.c_int32, C.POINTER(_h)],
    "icp_chain_set_target_index": [_h, C.c_int32, _ip],
    "icp_chain_destroy": [_h],
    "icp_chain_run": [_h, C.c_int32, C.c_int32, _dp, C.POINTER(ChainIO)],
    "icp_chain_run_device": [_h, C.c_int32, C.c_int32, C.c_void_p, C.POINTER(ChainIO), C.c_int32],
    "icp_ctx_synchronize": [_h],
    "icp_chain_last_run_stats": [_h, _dp, _lp],
    "icp_chain_set_lookahead": [_h, C.c_int32],
    "icp_chain_last_run_rounds": [_h, _lp],
    "icp_chain_set_statistics": [_h, C.POINTER(ChainStatsParams)],
    "icp_chain_statistics": [_h, C.c_int32, C.c_int32, _dp, _lp, _dp, _dp, _dp, _dp],
    "icp_debug_philox": [_h, C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32, C.POINTER(C.c_uint32)],
    "icp_debug_fp64_peak": [_h, _dp],
    "icp_debug_dmma_sweep": [_h, C.c_int32, C.c_int32, C.c_int32, _dp],
    "icp_chain_profile": [_h, C.c_int32, C.c_int32, _dp, C.c_uint64, _dp, _lp],
    "icp_debug_time_closest_point": [_h, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, _dp],
    "icp_debug_l2_bandwidth": [_h, C.c_int64, _dp],
    "icp_debug_i8_gram": [_h, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, _dp],
    "icp_debug_factor": [_h, C.c_int32, C.c_int32, _dp, _dp, _dp, _dp, C.c_double, C.c_int32, _dp, _dp, _dp, _ip],
    "icp_debug_svd_factor": [_h, C.c_int32, C.c_int32, _dp, _dp, C.c_double, _dp, _ip],
    "icp_debug_chain_schedule": [_h, C.c_int32, _ip, _lp],
}
EXPORTED_SYMBOLS = sorted(list(_SIGS) + ["icp_stage_name"])

_LIB = None


def load():
    """Loads libicpcuda.so; raises (never falls back) when it has not been built."""
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is missing: build it with `python icp-proposal_b200/build.py` "
                              "(nvcc, sm_100a). There is no CPU fallback.")
        lib = C.CDLL(LIB_PATH)
        for name, args in _SIGS.items():
            fn = getattr(lib, name)
            fn.argtypes = args
            fn.restype = C.c_int32
        lib.icp_stage_name.argtypes = [C.c_int32]
        lib.icp_stage_name.restype = C.c_char_p
        _LIB = lib
    return _LIB


def last_error(ctx=None):
    buf = C.create_string_buffer(1024)
    load().icp_last_error(ctx, buf, 1024)
    return buf.value.decode(errors="replace")


def check(rc, ctx=None):
    if rc != OK:
        raise IcpCudaError(rc, last_error(ctx))


def dptr(a):
    return a.ctypes.data_as(_dp)


def iptr(a):
    return a.ctypes.data_as(_ip)


def f64(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.float64)
    return a if shape is None else a.reshape(shape)


def i32(a):
    return np.ascontiguousarray(a, dtype=np.int32)
