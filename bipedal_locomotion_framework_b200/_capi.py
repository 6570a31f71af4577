"""ctypes binding of include/blf_ccm.h.  The library is the product: if it is missing this module
raises -- there is no Python or CPU fallback."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libblf_ccm.so")

WRENCH, AUTODYN, CTRL, REGRESSOR = 1, 2, 4, 8
FULL = WRENCH | AUTODYN | CTRL
PATH_BULK, PATH_DIRECT64 = 1, 2

OK, ERR_INVALID_ARG, ERR_INVALID_HANDLE, ERR_CUDA, ERR_NO_DEVICE, ERR_NOT_INITIALIZED, ERR_NCCL = \
    0, -1, -2, -3, -4, -5, -6

# every symbol include/blf_ccm.h declares
SYMBOLS = [
    "blf_ccm_version", "blf_ccm_last_error", "blf_ccm_create", "blf_ccm_destroy",
    "blf_ccm_set_uniform_params", "blf_ccm_eval_batch_soa", "blf_ccm_wrench_vjp_soa",
    "blf_ccm_eval_batch_aos",
    "blf_ccm_eval_batch_host", "blf_ccm_set_host_chunk", "blf_ccm_set_host_threads",
    "blf_ccm_eval_surface_points",
    "blf_ccm_rollout_cost_argmin_soa", "blf_ccm_argmin_pairs", "blf_ccm_argmin_allgather_nccl",
    "blf_ccm_last_path", "blf_ccm_launch_count", "blf_ccm_device", "blf_ccm_sm_count",
    "blf_ccm_device_alloc", "blf_ccm_device_free", "blf_ccm_device_alloc_compressible",
    "blf_ccm_pointer_is_compressible", "blf_ccm_host_alloc", "blf_ccm_host_free",
    "blf_ccm_copy_h2d", "blf_ccm_copy_d2h", "blf_ccm_stream_synchronize",
    "blf_rls_advance_batch", "blf_rls_advance_host", "blf_ccm_rls_advance_contacts",
    "blf_sys_kinematics_euler_step_soa", "blf_sys_kinematics_dynamics_host", "blf_sys_kinematics_dynamics",
    "blf_sys_kinematics_integrate_host", "blf_ccm_rollout_integrate_cost", "blf_ccm_rollout_cost_vjp",
    "blf_ccm_generalized_force_soa", "blf_ccm_rollout_integrate_cost_host",
    "blf_sys_mass_matrix_solve", "blf_sys_floating_base_acceleration", "blf_sys_floating_base_euler_step",
    "blf_ccm_p2p_mailbox_create", "blf_ccm_p2p_mailbox_connect", "blf_ccm_argmin_exchange_p2p",
    "blf_ccm_p2p_mailbox_destroy", "blf_ccm_rollout_set_exchange",
]


class BlfCcmError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"blf_ccm error {code}: {msg}")
        self.code = code


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -m bipedal_locomotion_framework_b200.build` "
            "(nvcc, sm_100a).  There is no CPU fallback for the contact-model backend.")
    L = C.CDLL(LIB_PATH)
    vp, i64, u32, dbl, ci = C.c_void_p, C.c_int64, C.c_uint, C.c_double, C.c_int
    L.blf_ccm_version.restype = C.c_char_p
    L.blf_ccm_last_error.restype = C.c_char_p
    L.blf_ccm_create.argtypes = [ci, C.POINTER(vp)]
    L.blf_ccm_destroy.argtypes = [vp]
    L.blf_ccm_set_uniform_params.argtypes = [vp, dbl, dbl, dbl, dbl]
    L.blf_ccm_eval_batch_soa.argtypes = [vp, i64, vp, vp, u32, vp, vp, vp, vp, vp]
    L.blf_ccm_wrench_vjp_soa.argtypes = [vp, i64, vp, vp, vp, vp, vp, vp]
    L.blf_ccm_eval_batch_aos.argtypes = [vp, i64, vp, vp, vp, vp, u32, vp, vp, vp, vp, vp]
    L.blf_ccm_eval_batch_host.argtypes = [vp, i64, vp, vp, vp, vp, u32, vp, vp, vp, vp]
    L.blf_ccm_set_host_chunk.argtypes = [vp, i64]
    L.blf_ccm_set_host_threads.argtypes = [vp, ci]
    L.blf_ccm_eval_surface_points.argtypes = [vp, vp, vp, vp, i64, vp, vp, vp, vp]
    L.blf_ccm_rollout_cost_argmin_soa.argtypes = [vp, i64, i64, vp, vp, u32, vp, vp, vp, vp, vp,
                                                  i64, vp, vp, vp]
    L.blf_ccm_argmin_pairs.argtypes = [vp, ci, vp, vp, vp]
    L.blf_ccm_argmin_allgather_nccl.argtypes = [vp, vp, ci, vp, vp, vp, vp]
    u64 = C.c_uint64
    L.blf_ccm_device_alloc.argtypes = [vp, u64, C.POINTER(vp)]
    L.blf_ccm_device_free.argtypes = [vp, vp]
    L.blf_ccm_device_alloc_compressible.argtypes = [vp, u64, C.POINTER(vp), C.POINTER(ci)]
    L.blf_ccm_pointer_is_compressible.argtypes = [vp, vp, C.POINTER(ci)]
    L.blf_ccm_host_alloc.argtypes = [vp, u64, C.POINTER(vp)]
    L.blf_ccm_host_free.argtypes = [vp, vp]
    L.blf_ccm_copy_h2d.argtypes = [vp, vp, vp, u64, vp]
    L.blf_ccm_copy_d2h.argtypes = [vp, vp, vp, u64, vp]
    L.blf_ccm_stream_synchronize.argtypes = [vp, vp]
    L.blf_rls_advance_batch.argtypes = [vp, i64, ci, ci, vp, vp, vp, dbl, vp, vp, vp]
    L.blf_rls_advance_host.argtypes = [vp, i64, ci, ci, vp, vp, vp, dbl, vp, vp]
    L.blf_ccm_rls_advance_contacts.argtypes = [vp, i64, vp, vp, vp, vp, dbl, vp, vp, vp]
    L.blf_sys_kinematics_euler_step_soa.argtypes = [vp, i64, dbl, dbl, vp, vp, vp, vp]
    L.blf_sys_kinematics_dynamics_host.argtypes = [vp, i64, dbl, vp, vp, vp, vp]
    L.blf_sys_kinematics_dynamics.argtypes = [vp, i64, dbl, vp, vp, vp, vp, vp]
    L.blf_sys_kinematics_integrate_host.argtypes = [vp, i64, dbl, dbl, dbl, ci, vp, vp, vp, i64,
                                                    vp, vp]
    L.blf_ccm_rollout_integrate_cost.argtypes = [vp, i64, ci, ci, dbl, dbl, vp, vp, vp, vp, vp, u32,
                                                 vp, vp, vp, vp, vp, vp, vp, i64, vp, vp, vp]
    L.blf_ccm_rollout_cost_vjp.argtypes = [vp, i64, ci, ci, dbl, dbl, vp, vp, vp, vp, vp, vp, vp, vp,
                                           vp, vp, vp, vp, vp, vp]
    L.blf_ccm_rollout_integrate_cost_host.argtypes = [vp, i64, ci, ci, dbl, dbl, vp, vp, vp, vp, vp,
                                                      vp, vp, vp, vp, vp]
    L.blf_ccm_generalized_force_soa.argtypes = [vp, i64, ci, ci, vp, vp, vp, vp, vp, vp, vp]
    L.blf_sys_mass_matrix_solve.argtypes = [vp, i64, ci, vp, vp, vp, vp, vp, vp]
    L.blf_sys_floating_base_acceleration.argtypes = [vp, i64, ci, ci, vp, vp, vp, vp, vp, vp, vp, vp,
                                                     vp, vp]
    L.blf_sys_floating_base_euler_step.argtypes = [vp, i64, ci, dbl, dbl, vp, vp, vp, vp, vp, vp]
    L.blf_ccm_p2p_mailbox_create.argtypes = [vp, ci, ci, vp]
    L.blf_ccm_p2p_mailbox_connect.argtypes = [vp, vp]
    L.blf_ccm_argmin_exchange_p2p.argtypes = [vp, vp, vp, vp]
    L.blf_ccm_p2p_mailbox_destroy.argtypes = [vp]
    L.blf_ccm_rollout_set_exchange.argtypes = [vp, vp]
    L.blf_ccm_last_path.argtypes = [vp]
    L.blf_ccm_launch_count.argtypes = [vp]
    L.blf_ccm_launch_count.restype = i64
    L.blf_ccm_device.argtypes = [vp]
    L.blf_ccm_sm_count.argtypes = [vp]
    _lib = L
    return L


def check(rc: int):
    if rc != 0:
        raise BlfCcmError(rc, lib().blf_ccm_last_error().decode())
