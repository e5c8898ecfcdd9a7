"""ctypes loader of libtds_b200.so (in-tree build, see build.py).  Fails loudly when missing."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


class LibraryMissing(RuntimeError):
    pass


def lib_path():
    # TDS_B200_LIB: an alternative in-tree build of the same library (A/B experiments of kernel variants)
    return os.environ.get("TDS_B200_LIB") or os.path.join(_HERE, "libtds_b200.so")


class CudaFunctionMetaData(ctypes.Structure):
    _fields_ = [("output_dim", ctypes.c_int), ("input_dim", ctypes.c_int), ("global_dim", ctypes.c_int)]


def lib():
    global _LIB
    if _LIB is not None:
        return _LIB
    path = lib_path()
    if not os.path.exists(path):
        raise LibraryMissing(
            f"{path} not found: build it with `python tiny-differentiable-simulator_b200/build.py` "
            "(there is no CPU / PyTorch fallback for the hot path)")
    L = ctypes.CDLL(path)
    dp = ctypes.POINTER(ctypes.c_double)
    fp = ctypes.c_void_p  # device or host float pointers are passed as raw addresses
    vp = ctypes.c_void_p
    ci = ctypes.c_int
    cd = ctypes.c_double
    L.tds_b200_last_error.restype = ctypes.c_char_p
    L.tds_b200_urdf_to_model.restype = ci
    L.tds_b200_urdf_to_model.argtypes = [ctypes.c_char_p, ctypes.c_char_p, ci, dp, ci]
    L.tds_b200_create.restype = vp
    L.tds_b200_create.argtypes = [dp, ci, ci, ci]
    L.tds_b200_destroy.argtypes = [vp]
    L.tds_b200_set_params.restype = ci
    L.tds_b200_set_params.argtypes = [vp, cd, dp, cd, cd, cd, cd, ci, ci]
    L.tds_b200_set_contact_model.restype = ci
    L.tds_b200_set_contact_model.argtypes = [vp, ci, cd, cd, cd, cd, ci]
    L.tds_b200_set_env.restype = ci
    L.tds_b200_set_env.argtypes = [vp, ci, dp, ci, cd, cd, cd, cd, ci]
    L.tds_b200_set_auto_reset.restype = ci
    L.tds_b200_set_auto_reset.argtypes = [vp, ci, dp]
    L.tds_b200_set_precision.restype = ci
    L.tds_b200_set_precision.argtypes = [vp, ci]
    L.tds_b200_env_reset_device.restype = ci
    L.tds_b200_env_reset_device.argtypes = [vp, vp, vp, ctypes.c_float, ctypes.c_ulonglong, ci, vp]
    L.tds_b200_env_rollout_device.restype = ci
    L.tds_b200_env_rollout_device.argtypes = [vp, vp, ci, ci, ctypes.c_float, vp, vp, vp]
    L.tds_b200_env_rollout_host.restype = ci
    L.tds_b200_env_rollout_host.argtypes = [vp, vp, ci, ci, ctypes.c_double, vp, ctypes.c_double, ctypes.c_ulonglong, ci, vp, vp]
    L.tds_b200_env_set_obs_stats.restype = ci
    L.tds_b200_env_set_obs_stats.argtypes = [vp, vp]
    L.tds_b200_ars_perturb_device.restype = ci
    L.tds_b200_ars_perturb_device.argtypes = [vp, vp, vp, ctypes.c_float, vp, ci, vp]
    L.tds_b200_ars_update_device.restype = ci
    L.tds_b200_ars_update_device.argtypes = [vp, vp, vp, vp, vp, ctypes.c_float, ctypes.c_float, ci, vp]
    L.tds_b200_num_visuals.restype = ci
    L.tds_b200_num_visuals.argtypes = [vp]
    L.tds_b200_env_step_visual_device.restype = ci
    L.tds_b200_env_step_visual_device.argtypes = [vp, vp, vp, vp, vp, vp, vp]
    L.tds_b200_get_precision.restype = ci
    L.tds_b200_get_precision.argtypes = [vp]
    L.tds_b200_validate_model.restype = ci
    L.tds_b200_validate_model.argtypes = [ctypes.POINTER(ctypes.c_double), ci]
    L.tds_b200_kernel_name.restype = ctypes.c_char_p
    L.tds_b200_kernel_name.argtypes = [vp]
    L.tds_b200_get_dims.restype = ci
    L.tds_b200_get_dims.argtypes = [vp, ctypes.POINTER(ci)]
    L.tds_b200_step_device.restype = ci
    L.tds_b200_step_device.argtypes = [vp, ci, ci] + [fp] * 10 + [vp]
    L.tds_b200_step_host.restype = ci
    L.tds_b200_step_host.argtypes = [vp, ci, ci, dp, dp, dp, dp, dp, dp, dp]
    L.tds_b200_jacobian_dims.restype = ci
    L.tds_b200_jacobian_dims.argtypes = [vp, ci, ci, ctypes.POINTER(ci)]
    L.tds_b200_step_jacobian_device.restype = ci
    L.tds_b200_step_jacobian_device.argtypes = [vp, ci, ci, fp, fp, fp, vp, vp]
    L.tds_b200_step_jacobian_host.restype = ci
    L.tds_b200_step_jacobian_host.argtypes = [vp, ci, ci, dp, dp, dp, dp]
    L.tds_b200_step_jvp_device.restype = ci
    L.tds_b200_step_jvp_device.argtypes = [vp, ci, ci, fp, fp, fp, vp, vp, vp, vp, vp]
    L.tds_b200_step_vjp_device.restype = ci
    L.tds_b200_step_vjp_device.argtypes = [vp, ci, ci, fp, fp, fp, vp, vp, vp, vp, vp]
    L.tds_b200_integrate_euler_device.restype = ci
    L.tds_b200_integrate_euler_device.argtypes = [vp, fp, fp, fp, vp]
    L.tds_b200_integrate_euler_qdd_device.restype = ci
    L.tds_b200_integrate_euler_qdd_device.argtypes = [vp, fp, fp, vp]
    L.tds_b200_model_contact_pairs.restype = ci
    L.tds_b200_model_contact_pairs.argtypes = [dp, ci, vp, ci]
    L.tds_b200_contact_pairs.restype = ci
    L.tds_b200_contact_pairs.argtypes = [vp, vp, ci]
    L.tds_b200_contact_list_device.restype = ci
    L.tds_b200_contact_list_device.argtypes = [vp, fp, vp, vp, vp]
    L.tds_b200_contact_list_host.restype = ci
    L.tds_b200_contact_list_host.argtypes = [vp, vp, vp]
    L.tds_b200_rigid_create.restype = vp
    L.tds_b200_rigid_create.argtypes = [vp, ci, ci, ci]
    L.tds_b200_rigid_destroy.restype = None
    L.tds_b200_rigid_destroy.argtypes = [vp]
    L.tds_b200_rigid_set_params.restype = ci
    L.tds_b200_rigid_set_params.argtypes = [vp, ctypes.c_double, vp, ctypes.c_double, ctypes.c_double, ctypes.c_double, ci]
    L.tds_b200_rigid_step_device.restype = ci
    L.tds_b200_rigid_step_device.argtypes = [vp, vp, vp, vp, ci, vp]
    L.tds_b200_rigid_step_host.restype = ci
    L.tds_b200_rigid_step_host.argtypes = [vp, vp, vp, ci, vp]
    L.tds_b200_rigid_jacobian_host.restype = ci
    L.tds_b200_rigid_jacobian_host.argtypes = [vp, vp, vp, ci, vp, vp]
    L.tds_b200_rigid_jvp_device.restype = ci
    L.tds_b200_rigid_jvp_device.argtypes = [vp, vp, vp, ci, vp, vp, vp, vp]
    L.tds_b200_rigid_vjp_device.restype = ci
    L.tds_b200_rigid_vjp_device.argtypes = [vp, vp, vp, ci, vp, vp, vp, vp]
    L.tds_b200_contact_tuples.restype = ci
    L.tds_b200_contact_tuples.argtypes = [vp, vp, ci]
    L.tds_b200_model_contact_tuples.restype = ci
    L.tds_b200_model_contact_tuples.argtypes = [vp, ci, vp, ci]
    L.tds_b200_contact_list_candidates_host.restype = ci
    L.tds_b200_contact_list_candidates_host.argtypes = [vp, vp, vp]
    L.tds_b200_env_set_state_host.restype = ci
    L.tds_b200_env_set_state_host.argtypes = [vp, dp, dp]
    L.tds_b200_env_get_state_host.restype = ci
    L.tds_b200_env_get_state_host.argtypes = [vp, dp, dp]
    L.tds_b200_env_step_host.restype = ci
    L.tds_b200_env_step_host.argtypes = [vp, fp, fp, fp, fp]
    L.tds_b200_env_step_device.restype = ci
    L.tds_b200_env_step_device.argtypes = [vp, fp, fp, fp, vp]
    L.tds_b200_stream.restype = vp
    L.tds_b200_stream.argtypes = [vp]
    L.tds_b200_env_q.restype = vp
    L.tds_b200_env_q.argtypes = [vp]
    L.tds_b200_env_qd.restype = vp
    L.tds_b200_env_qd.argtypes = [vp]
    L.cuda_model_laikago_forward_zero.argtypes = [ci, ci, ci, dp, dp]
    L.cuda_model_laikago_forward_zero_meta.restype = CudaFunctionMetaData
    L.cuda_model_laikago_forward_zero_allocate.argtypes = [ci]
    L.cuda_model_ant_forward_zero.argtypes = [ci, ci, ci, dp, dp]
    L.cuda_model_ant_forward_zero_meta.restype = CudaFunctionMetaData
    L.cuda_model_ant_forward_zero_allocate.argtypes = [ci]
    _LIB = L
    return L


def last_error():
    return lib().tds_b200_last_error().decode()


# every symbol include/tds_b200.h declares (checked by the CPU test-suite)
DECLARED_SYMBOLS = [
    "tds_b200_last_error", "tds_b200_urdf_to_model", "tds_b200_create", "tds_b200_destroy",
    "tds_b200_set_params", "tds_b200_set_contact_model", "tds_b200_set_env", "tds_b200_set_auto_reset", "tds_b200_validate_model", "tds_b200_set_precision", "tds_b200_get_precision", "tds_b200_kernel_name", "tds_b200_get_dims", "tds_b200_env_reset_device",
    "tds_b200_env_set_obs_stats", "tds_b200_ars_perturb_device", "tds_b200_ars_update_device", "tds_b200_env_rollout_device", "tds_b200_env_rollout_host", "tds_b200_num_visuals", "tds_b200_env_step_visual_device",
    "model_info", "b200_laikago_forward_zero", "b200_laikago_forward_zero_meta", "b200_laikago_forward_zero_allocate",
    "b200_laikago_forward_zero_deallocate", "b200_laikago_forward_zero_send_local", "b200_laikago_forward_zero_send_global",
    "b200_laikago_jacobian", "b200_laikago_jacobian_meta", "b200_laikago_jacobian_allocate", "b200_laikago_jacobian_deallocate",
    "b200_laikago_jacobian_send_local", "b200_laikago_jacobian_send_global",
    "tds_b200_jacobian_dims", "tds_b200_step_jacobian_device", "tds_b200_step_jacobian_host", "tds_b200_step_jvp_device", "tds_b200_step_vjp_device", "tds_b200_integrate_euler_device", "tds_b200_integrate_euler_qdd_device", "tds_b200_contact_pairs", "tds_b200_model_contact_pairs", "tds_b200_contact_tuples", "tds_b200_model_contact_tuples", "tds_b200_contact_list_device", "tds_b200_contact_list_host", "tds_b200_contact_list_candidates_host",
    "tds_b200_rigid_create", "tds_b200_rigid_destroy", "tds_b200_rigid_set_params", "tds_b200_rigid_step_device", "tds_b200_rigid_step_host", "tds_b200_rigid_jacobian_host", "tds_b200_rigid_jvp_device", "tds_b200_rigid_vjp_device",
    "tds_b200_step_device", "tds_b200_step_host", "tds_b200_env_set_state_host",
    "tds_b200_env_get_state_host", "tds_b200_env_step_host", "tds_b200_env_step_device",
    "tds_b200_stream", "tds_b200_env_q", "tds_b200_env_qd", "cuda_model_laikago_forward_zero",
    "cuda_model_laikago_forward_zero_meta", "cuda_model_laikago_forward_zero_allocate",
    "cuda_model_laikago_forward_zero_deallocate",
    "cuda_model_ant_forward_zero", "cuda_model_ant_forward_zero_meta", "cuda_model_ant_forward_zero_allocate",
    "cuda_model_ant_forward_zero_deallocate",
]
