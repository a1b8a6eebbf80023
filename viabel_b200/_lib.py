"""ctypes binding of libviabel_b200.so (the C ABI declared in include/viabel_b200.h).

The product path has no CPU fallback: importing this module fails loudly when the
shared library has not been built (`python viabel_b200/csrc/build.py`), and every compute
entry point needs CUDA device pointers.
"""
import ctypes
import os
from ctypes import c_char_p, c_double, c_int, c_int64, c_size_t, c_uint64, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
# VIABEL_B200_LIB points at another build of the same library (A/B runs of kernel variants)
LIB_PATH = os.environ.get('VIABEL_B200_LIB') or os.path.join(_HERE, 'libviabel_b200.so')

VB_OK = 0
VB_ERR_INVALID_ARG, VB_ERR_UNSUPPORTED, VB_ERR_CUDA, VB_ERR_WORKSPACE, VB_ERR_NUMERIC = -1, -2, -3, -4, -5
FAMILY_MF_GAUSSIAN, FAMILY_MF_STUDENT = 0, 1
LINK_LOGISTIC, LINK_PROBIT, LINK_GAUSSIAN = 0, 1, 2
OBJ_EXCLUSIVE_KL, OBJ_EXCLUSIVE_KL_PATH, OBJ_ALPHA = 0, 1, 2

if not os.path.exists(LIB_PATH):
    raise ImportError(
        'viabel_b200: %s is missing. Build it with `python viabel_b200/csrc/build.py` '
        '(nvcc, sm_100a). There is no CPU fallback.' % LIB_PATH)

lib = ctypes.CDLL(LIB_PATH)

P = c_void_p
_PROTOS = {
    'vb_last_error': (c_char_p, []),
    'vb_version': (c_int, []),
    'vb_device_sm_count': (c_int, []),
    'vb_philox_normal_f64': (c_int, [P, c_int64, c_uint64, c_uint64, c_int, P]),
    'vb_philox_normal_f32': (c_int, [P, c_int64, c_uint64, c_uint64, c_int, P]),
    'vb_philox_chisquare_f64': (c_int, [P, c_int64, c_double, c_uint64, c_uint64, P]),
    'vb_philox_student_t_f64': (c_int, [P, c_int64, c_double, c_uint64, c_uint64, c_int, P]),
    'vb_mf_sample_f64': (c_int, [P, P, P, c_int64, c_int, P]),
    'vb_mf_log_density_f64': (c_int, [P, P, c_int64, c_int, c_int, c_double, P, P]),
    'vb_glm_sweep_workspace_bytes': (c_size_t, [c_int64, c_int, c_int64]),
    'vb_glm_sweep_f64': (c_int, [P, c_int64, P, c_int64, c_int, c_int, P, P, P, P, c_int64, c_int,
                                 P, P, P, P, c_size_t, P]),
    'vb_mf_alpha_weights_f64': (c_int, [P, P, P, P, c_int64, c_int, c_int, c_double, c_double, c_double,
                                        P, P, P, P]),
    'vb_mf_objective_finish_workspace_bytes': (c_size_t, [c_int64]),
    'vb_mf_objective_finish_f64': (c_int, [P, P, P, P, P, P, P, c_int64, c_int, c_int, c_double, c_double,
                                           c_int, c_double, P, P, P, P, c_size_t, P]),
    'vb_rmsprop_step_f64': (c_int, [P, P, P, P, c_int64, c_double, c_double, c_double, c_int, P]),
    'vb_adam_step_f64': (c_int, [P, P, P, P, P, c_int64, c_double, c_double, c_double, c_double, c_int, P]),
    'vb_glm_fast_model_bytes': (c_size_t, [c_int64, c_int]),
    'vb_glm_fast_workspace_bytes': (c_size_t, [c_int64, c_int, c_int64]),
    'vb_glm_fast_create': (c_int, [P, P, c_int64, P, c_int64, c_int, c_int, P, c_size_t, P, P]),
    'vb_glm_fast_destroy': (c_int, [P]),
    'vb_glm_fast_sweep': (c_int, [P, P, P, P, c_int64, c_int, P, P, P, P, c_size_t, P, P]),
    'vb_psis_workspace_bytes': (c_size_t, [c_int64, c_double]),
    'vb_psis_tail_capacity': (c_int64, [c_int64, c_double]),
    'vb_psislw_f64': (c_int, [P, P, c_int64, c_double, c_int, P, P, P, P, c_size_t, P]),
    'vb_psis_batch_max_n': (c_int64, [c_double]),
    'vb_psislw_batch_f64': (c_int, [P, c_int64, c_int64, c_int64, c_double, P, c_int64, P, P, P, P]),
    'vb_psis_dist_workspace_bytes': (c_size_t, [c_int64, c_int64, c_double, c_int]),
    'vb_psis_dist_record_doubles': (c_int64, [c_int64, c_double]),
    'vb_psis_dist_local': (c_int, [P, c_int64, c_int64, c_int64, c_double, c_int, c_int, P, P, c_size_t, P]),
    'vb_psis_dist_global': (c_int, [P, c_int64, c_int64, c_double, c_int, P, P, c_size_t, P]),
    'vb_psis_dist_apply': (c_int, [P, P, c_int64, c_int64, c_int64, c_double, c_int, c_int, P, P, c_size_t, P]),
    'vb_divergence_moments_f64': (c_int, [P, c_int64, c_double, P, P]),
    'vb_mf_reduce_grads_f64': (c_int, [P, P, P, c_int64, c_int, P, P, P]),
    'vb_glm_link_workspace_bytes': (c_size_t, [c_int64, c_int]),
    'vb_glm_link_f64': (c_int, [P, P, c_int64, c_int, c_int, P, P, c_size_t, P]),
    'vb_target_logp_grad_f64': (c_int, [P, c_int64, c_int, c_int, P, P, c_double, c_double, P, P, P]),
    'vb_glm_point_workspace_bytes': (c_size_t, [c_int64, c_int, c_int, c_int]),
    'vb_glm_point_f64': (c_int, [P, c_int64, P, c_int64, c_int, c_int, P, P, c_int, P, P, P, P, P, c_size_t, P]),
    'vb_sample_moments_workspace_bytes': (c_size_t, [c_int64, c_int, c_int]),
    'vb_sample_moments_f64': (c_int, [P, c_int64, c_int, c_int64, P, P, P, P, P, c_size_t, P]),
    'vb_faso_rhat_workspace_bytes': (c_size_t, [c_int, c_int]),
    'vb_faso_rhat_f64': (c_int, [P, c_int64, c_int, c_int64, P, c_int, c_double, P, P, c_size_t, P]),
    'vb_ring_mean_f64': (c_int, [P, c_int64, c_int, c_int64, c_int64, P, P, P]),
    'vb_faso_center_f64': (c_int, [P, c_int64, c_int, c_int64, c_int64, c_int64, P, P, P]),
    'vb_faso_ess_f64': (c_int, [P, c_int64, c_double, c_int64, c_int, P, P]),
    'vb_dis_bisection_f64': (c_int, [P, P, P, c_int64, c_double, c_double, c_double, c_int, P, P, P]),
    'vb_mf_score_workspace_bytes': (c_size_t, [c_int]),
    'vb_mf_score_f64': (c_int, [P, P, P, P, c_double, c_int64, c_int, c_int, c_double, P, P, P, c_size_t, P]),
    'vb_mvt_score_workspace_bytes': (c_size_t, [c_int64, c_int]),
    'vb_mvt_score_f64': (c_int, [P, P, P, P, c_double, c_int64, c_int, c_double, P, P, P, c_size_t, P]),
    'vb_lr_score_workspace_bytes': (c_size_t, [c_int64, c_int, c_int]),
    'vb_lr_score_f64': (c_int, [P, P, P, P, P, c_double, c_int64, c_int, c_int, P, P, P, c_size_t, P]),
    'vb_mf_target_log_weights_f64': (c_int, [P, c_int64, c_int, c_int, c_double, c_uint64, c_uint64, c_int, c_int, P, P,
                                             c_double, P, P, P]),
    'vb_gemm_f64': (c_int, [c_int, c_int, c_int, c_int, c_int, c_double, P, c_int64, P, c_int64, P, c_int64, P, P, P, P, P, P]),
    'vb_mvt_unpack_f64': (c_int, [P, c_int, P, P, P]),
    'vb_mvt_sigma_f64': (c_int, [P, c_int, c_double, P, P]),
    'vb_mvt_transform_workspace_bytes': (c_size_t, [c_int, c_int]),
    'vb_mvt_transform_f64': (c_int, [P, P, P, c_double, c_int, c_int, P, P, P, P, P, P, c_size_t, P]),
    'vb_mvt_objective_workspace_bytes': (c_size_t, [c_int, c_int]),
    'vb_mvt_path_workspace_bytes': (c_size_t, [c_int, c_int]),
    'vb_mvt_objective_f64': (c_int, [P, P, P, P, P, P, P, P, c_int, c_int, c_double, c_int, c_double, P, P, P, c_size_t, P]),
    'vb_mvt_log_density_workspace_bytes': (c_size_t, [c_int64, c_int]),
    'vb_mvt_log_density_f64': (c_int, [P, P, P, P, c_int64, c_int, c_double, P, P, c_size_t, P]),
    'vb_mvt_chol_transform_f64': (c_int, [P, P, P, c_double, c_int, c_int, P, P, P, P]),
    'vb_mvt_chol_objective_workspace_bytes': (c_size_t, [c_int, c_int]),
    'vb_mvt_chol_path_workspace_bytes': (c_size_t, [c_int, c_int]),
    'vb_mvt_chol_objective_f64': (c_int, [P, P, P, P, P, P, c_int, c_int, c_double, c_int, c_double, P, P, P, c_size_t, P]),
    'vb_mvt_target_log_weights_workspace_bytes': (c_size_t, [c_int]),
    'vb_mvt_target_log_weights_f64': (c_int, [P, P, c_int64, c_int64, c_int64, c_int, c_double, c_uint64, c_uint64, c_int,
                                              P, P, c_double, P, P, P, c_size_t, P]),
    'vb_lr_target_log_weights_workspace_bytes': (c_size_t, [c_int, c_int]),
    'vb_lr_target_log_weights_f64': (c_int, [P, P, c_int64, c_int64, c_int64, c_int, c_int, c_uint64, c_uint64, c_int,
                                             P, P, c_double, P, P, P, c_size_t, P]),
    'vb_hier_workspace_bytes': (c_size_t, [c_int, c_int]),
    'vb_hier_logp_grad_f64': (c_int, [P, P, P, c_int64, c_int, c_int, P, c_int, P, P, P, c_size_t, P]),
    # peer-memory communicator and the fused step (structures: viabel_b200/engine.py)
    'vb_comm_create': (c_int, [P, c_int, c_int, c_size_t, P]),
    'vb_comm_connect': (c_int, [P, P]),
    'vb_comm_connect_ptrs': (c_int, [P, P]),
    'vb_comm_buffer': (c_void_p, [P]),
    'vb_comm_allreduce_sum_f64': (c_int, [P, P, c_int64, P]),
    'vb_comm_error': (c_int, [P]),
    'vb_comm_destroy': (c_int, [P]),
    'vb_mf_step_workspace_bytes': (c_size_t, [c_int, c_int]),
    'vb_mf_step_glm': (c_int, [P, P, P, P, P, c_size_t, P]),
}

#: symbols declared in include/viabel_b200.h that this build exports
EXPORTED = []
for _name, (_res, _args) in _PROTOS.items():
    _fn = getattr(lib, _name)          # AttributeError here = header/library mismatch
    _fn.restype = _res
    _fn.argtypes = _args
    EXPORTED.append(_name)


def last_error():
    return lib.vb_last_error().decode('utf-8', 'replace')


def check(rc):
    """Map a C-ABI status to the exception class the reference raises."""
    if rc == VB_OK:
        return
    msg = last_error()
    if rc in (VB_ERR_INVALID_ARG, VB_ERR_NUMERIC):
        raise ValueError(msg)
    if rc == VB_ERR_UNSUPPORTED:
        raise NotImplementedError(msg)
    raise RuntimeError('viabel_b200 [%d]: %s' % (rc, msg))


def ptr(t):
    """Device pointer of a torch tensor (None -> NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError('viabel_b200: expected a CUDA tensor; there is no CPU path')
    if not t.is_contiguous():
        raise RuntimeError('viabel_b200: expected a contiguous tensor')
    return c_void_p(t.data_ptr())


def stream():
    import torch
    return c_void_p(torch.cuda.current_stream().cuda_stream)
