"""ctypes binding of libpiml_b200.so (the C ABI declared in include/piml_b200.h).

The product path has NO CPU fallback: if the library is missing, or an entry point is called without a CUDA device,
this module raises -- it never routes to the oracle or to eager PyTorch.
"""
import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libpiml_b200.so")

_lib = None

vp, i32, i64, f32 = C.c_void_p, C.c_int, C.c_int64, C.c_float

# Linears the PINNSF backward's dW launch can take (DW_MAX_JOBS in csrc/mlp_bwd.cu; keep the two equal).
PINNSF_DW_JOBS = 38


class MlapmParams(C.Structure):
    """piml_mlapm_params"""
    _fields_ = [("version", i32), ("tau", f32), ("A", f32), ("B", f32), ("C", f32), ("D", f32),
                ("theta_deg", f32), ("exact_math", i32)]


class NetDesc(C.Structure):
    """piml_net_desc"""
    _fields_ = [("n_enc", i32), ("enc_dims", i32 * 9), ("proc_mode", i32), ("n_dec", i32), ("dec_dims", i32 * 9),
                ("n_coll", i32), ("coll_dims", i32 * 5), ("kind", i32)]


class RolloutArgs(C.Structure):
    """piml_rollout_args"""
    _fields_ = [("desc", C.POINTER(NetDesc)), ("packed", vp), ("packed_tc", vp), ("has_obs", i32), ("tau", f32),
                ("S", i32), ("N", i32), ("M", i32), ("D", i32), ("T", i32), ("t_start", i32), ("dt", f32),
                ("kp", i32), ("cos_p", f32), ("thr_p", f32), ("ko", i32), ("cos_o", f32), ("thr_o", f32),
                ("obstacles", vp), ("obs_per_scene", i32),
                ("pos_tm", vp), ("vel_tm", vp), ("acc_tm", vp), ("dest_tm", vp), ("dest_idx_tm", vp),
                ("entry_tm", vp), ("dest_num", vp), ("waypoints", vp), ("desired_speed", vp),
                ("p", vp), ("v", vp), ("a", vp), ("dest", vp), ("dest_idx", vp), ("hist_v", vp),
                ("ped_f", vp), ("obs_f", vp), ("self_f", vp), ("dest_f", vp), ("a_next", vp),
                ("rec_p", vp), ("rec_v", vp), ("rec_a", vp), ("rec_mask", vp), ("sfm", vp)]


class SfmSweepArgs(C.Structure):
    """piml_sfm_sweep_args"""
    _fields_ = [("S", i32), ("N", i32), ("M", i32), ("D", i32), ("T", i32), ("t_start", i32), ("dt", f32),
                ("kp", i32), ("cos_p", f32), ("thr_p", f32), ("ko", i32), ("cos_o", f32), ("thr_o", f32),
                ("obstacles", vp), ("pos_tm", vp), ("vel_tm", vp), ("acc_tm", vp), ("dest_tm", vp),
                ("dest_idx_tm", vp), ("entry_tm", vp), ("mask_p", vp), ("dest_num", vp), ("waypoints", vp),
                ("desired_speed", vp), ("p", vp), ("v", vp), ("a", vp), ("dest", vp), ("dest_idx", vp),
                ("ped_f", vp), ("obs_f", vp), ("self_f", vp), ("params", vp), ("err_sum", vp), ("err_count", vp),
                ("rec_p", vp), ("rec_v", vp), ("rec_a", vp), ("rec_mask", vp), ("workspace", vp),
                ("workspace_bytes", i64)]


class NnStepArgs(C.Structure):
    """piml_nn_step_args"""
    _fields_ = [("desc", C.POINTER(NetDesc)), ("packed_tc", vp), ("has_obs", i32), ("tau", f32),
                ("S", i32), ("N", i32), ("M", i32), ("D", i32), ("dt", f32), ("remove_on_arrival", i32),
                ("kp", i32), ("cos_p", f32), ("thr_p", f32), ("ko", i32), ("cos_o", f32), ("thr_o", f32),
                ("obstacles", vp), ("obs_per_scene", i32), ("dest_num", vp), ("waypoints", vp), ("desired_speed", vp),
                ("p", vp), ("v", vp), ("a", vp), ("dest", vp), ("dest_idx", vp), ("hist_v", vp),
                ("entry", vp), ("p_gt", vp), ("v_gt", vp), ("a_gt", vp), ("dest_gt", vp), ("dest_idx_gt", vp),
                ("rec_p", vp), ("rec_v", vp), ("rec_a", vp), ("rec_mask", vp), ("a_next", vp),
                ("ped_f", vp), ("obs_f", vp), ("self_f", vp), ("dest_f", vp)]


class SfmParams(C.Structure):
    """piml_sfm_params"""
    _fields_ = [("A_ped", f32), ("B_ped", f32), ("A_obs", f32), ("B_obs", f32), ("eps", f32), ("tau", f32)]


# name -> (restype, argtypes); must list every symbol include/piml_b200.h declares (tests check this).
SIGNATURES = {
    "piml_version": (i32, []),
    "piml_last_error": (C.c_char_p, []),
    "piml_launch_count": (i64, []),
    "piml_device_info": (i32, [C.POINTER(i32), C.POINTER(i32)]),
    "piml_pipe_probe": (i32, [i32, i32, i32, vp, vp]),
    "piml_heading_f32": (i32, [vp, i32, i32, i32, vp, vp]),
    "piml_desired_speed_f32": (i32, [vp, i32, i32, i32, vp, vp]),
    "piml_relative_quantity_f32": (i32, [vp, vp, i64, i32, i32, i32, vp, vp]),
    "piml_filtered_features_f32": (i32, [vp, vp, vp, i64, i32, i32, i32, f32, vp, vp]),
    "piml_select_neighbors_f32": (i32, [vp, vp, i64, vp, i32, i32, i32, i32, f32, vp, vp, vp]),
    "piml_relative_features_f32": (i32, [vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, f32, f32, i32, f32,
                                         f32, vp, vp, vp, vp, vp, vp, vp, vp]),
    "piml_state_features_f32": (i32, [vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, f32, f32, i32, f32, f32, vp, vp,
                                      vp, vp, vp, vp, vp]),
    "piml_state_features_rows_f32": (i32, [vp, vp, vp, vp, vp, i32, i32, i64, i64, i32, f32, f32, i32, f32, f32, vp,
                                           vp, vp, vp, vp, vp, vp]),
    "piml_collision_label_f32": (i32, [vp, i64, vp, vp]),
    "piml_set_feature_algorithm": (i32, [i32]),
    "piml_free_workspace": (i32, []),
    "piml_mlapm_workspace_bytes": (i64, [i64]),
    "piml_mlapm_step_f32": (i32, [vp, vp, vp, i32, vp, i64, i64, i64, C.POINTER(MlapmParams), f32, vp, vp, vp]),
    "piml_mlapm_advance_f32": (i32, [vp, vp, vp, i32, vp, i64, i64, i64, C.POINTER(MlapmParams), f32, f32, vp, vp,
                                     vp, vp, vp]),
    "piml_mlapm_workspace_bytes_sym": (i64, [i64]),
    "piml_set_mlapm_algorithm": (i32, [i32]),
    "piml_mlapm_cull_radius": (f32, [C.POINTER(MlapmParams)]),
    "piml_mlapm_cull_items": (i32, [vp, i64, C.POINTER(i64)]),
    "piml_mlapm_advance_ws_f32": (i32, [vp, vp, vp, i32, vp, i64, i64, i64, C.POINTER(MlapmParams), f32, f32, vp, vp,
                                        vp, vp, i64, vp]),
    "piml_mlapm_scenes_advance_f32": (i32, [vp, vp, vp, i32, vp, vp, i64, i64, C.POINTER(MlapmParams), vp, f32, f32,
                                            vp, vp, vp, vp]),
    "piml_scatter_rows_push_f32": (i32, [vp, vp, vp, i64, i64, i32, vp, vp, vp, vp]),
    "piml_mlapm_sym_shard_rows": (i32, [i64, i32, i32, C.POINTER(i64), C.POINTER(i64)]),
    "piml_mlapm_sym_inbox_bytes": (i64, [i64, i32]),
    "piml_mlapm_sym_shard_workspace_bytes": (i64, [i64, i32]),
    "piml_mlapm_sym_pairs_push_f32": (i32, [vp, vp, vp, i64, i32, i32, C.POINTER(MlapmParams), vp, vp, i64, vp]),
    "piml_mlapm_sym_finalize_push_f32": (i32, [vp, vp, vp, i32, vp, i64, i32, i32, C.POINTER(MlapmParams), f32, f32,
                                               vp, vp, vp, vp, vp, i64, vp]),
    "piml_mlapm_advance_push_f32": (i32, [vp, vp, vp, i32, vp, i64, i64, i64, C.POINTER(MlapmParams), f32, f32, i32,
                                          vp, vp, vp, vp, vp]),
    "piml_calc_acceleration_f32": (i32, [vp, i64, i32, i32, f32, f32, f32, f32, f32, f32, vp, vp]),
    "piml_rollout_losses_workspace_floats": (i64, [i32, i32]),
    "piml_rollout_losses_f32": (i32, [vp, vp, i64, i32, i32, i32, f32, i32, vp, vp, vp, vp, vp, vp]),
    "piml_rollout_losses_backward_f32": (i32, [vp, vp, i64, i32, i32, i32, f32, i32, vp, vp, vp, vp, vp, vp]),
    "piml_l1_sum_f32": (i32, [vp, i64, f32, vp, vp]),
    "piml_l1_sum_backward_f32": (i32, [vp, i64, f32, vp, vp, vp]),
    "piml_bce_sum_f32": (i32, [vp, vp, i64, vp, vp]),
    "piml_bce_sum_backward_f32": (i32, [vp, vp, i64, vp, vp, vp]),
    "piml_metrics_frames_f32": (i32, [vp, vp, vp, i32, i32, f32, i32, f32, i32, vp, vp, vp, vp, vp]),
    "piml_sfm_forward_f32": (i32, [C.POINTER(SfmParams), vp, vp, vp, i64, i32, i32, vp, vp, vp, vp]),
    "piml_pinnsf_packed_floats": (i64, [C.POINTER(NetDesc)]),
    "piml_pinnsf_pack_f32": (i32, [C.POINTER(NetDesc), vp, vp, vp]),
    "piml_pinnsf_forward_f32": (i32, [C.POINTER(NetDesc), vp, i32, f32, vp, vp, vp, i64, i32, i32, i32, vp, vp, vp,
                                      vp, vp, vp, vp]),
    "piml_tc_selftest_f32": (i32, [vp, vp, i32, i32, i32, vp, vp]),
    "piml_tc16_selftest_f32": (i32, [vp, vp, i32, i32, i32, i32, vp, vp]),
    "piml_pinnsf_packed_tc_floats": (i64, [C.POINTER(NetDesc)]),
    "piml_pinnsf_pack_tc_f32": (i32, [C.POINTER(NetDesc), vp, vp, vp]),
    "piml_pinnsf_forward_tc_f32": (i32, [C.POINTER(NetDesc), vp, i32, f32, vp, vp, vp, i64, i32, i32, i32, vp, vp, vp,
                                         vp]),
    "piml_pinnsf_stash_floats": (i64, [C.POINTER(NetDesc), i32, i64, i32, i32]),
    "piml_pinnsf_backward_workspace_floats": (i64, [C.POINTER(NetDesc), i32, i64, i32, i32]),
    "piml_pinnsf_forward_train_f32": (i32, [C.POINTER(NetDesc), vp, i32, f32, vp, vp, vp, i64, i32, i32, i32, vp, vp,
                                            vp, vp, vp, vp, vp, vp]),
    "piml_pinnsf_packed_bwd_floats": (i64, [C.POINTER(NetDesc)]),
    "piml_pinnsf_pack_bwd_f32": (i32, [C.POINTER(NetDesc), vp, vp, vp]),
    "piml_pinnsf_backward_f32": (i32, [C.POINTER(NetDesc), vp, i32, f32, vp, vp, vp, i64, i32, i32, i32, vp, vp, vp,
                                       vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]),
    "piml_relative_features_backward_f32": (i32, [vp, vp, vp, vp, i32, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp]),
    "piml_collision_detection_f32": (i32, [vp, vp, i32, i32, i32, f32, i32, vp, vp, vp]),
    "piml_rollout_f32": (i32, [C.POINTER(RolloutArgs), vp]),
    "piml_sfm_sweep_workspace_bytes": (i64, [C.POINTER(SfmSweepArgs)]),
    "piml_sfm_sweep_f32": (i32, [C.POINTER(SfmSweepArgs), vp]),
    "piml_nn_step_supported": (i32, [C.POINTER(NetDesc)]),
    "piml_nn_step_f32": (i32, [C.POINTER(NnStepArgs), vp]),
    "piml_nn_step_shard_f32": (i32, [C.POINTER(NnStepArgs), i64, i64, i32, vp, vp, vp, vp]),
    "piml_integrate_step_backward_f32": (i32, [vp, i64, f32, vp, vp, vp, vp, vp, vp, vp, vp]),
    "piml_integrate_step_f32": (i32, [vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, f32, i32, vp, vp, vp, vp, vp,
                                      vp, vp, vp, vp, vp, vp, vp]),
}


def load():
    """Load the shared library (no GPU needed for loading / symbol lookup)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -m piml_b200.build` (nvcc, sm_100a). "
                "piml_b200 has no CPU fallback.")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def last_error():
    return load().piml_last_error().decode()


def check(rc, what):
    if rc != 0:
        raise RuntimeError(f"{what} failed (code {rc}): {last_error()}")


def launch_count():
    return int(load().piml_launch_count())


def cuda_device():
    if not torch.cuda.is_available():
        raise RuntimeError("piml_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device())


def require_cuda(*tensors):
    """Every tensor argument of a compute entry point must live on one CUDA device."""
    cuda_device()
    dev = None
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise RuntimeError("piml_b200: expected CUDA tensors (move inputs with .cuda() first)")
        dev = dev or t.device
        if t.device != dev:
            raise RuntimeError("piml_b200: tensors on different devices")
    return dev


def stage(*tensors):
    """Host-buffer entry: returns (device, origin_device, [tensors on the device]).  CUDA tensors pass through;
    host tensors are copied to the current CUDA device (the reference's scripts hand over CPU tensors).  The compute
    itself always runs in libpiml_b200.so on the GPU."""
    first = next(t for t in tensors if t is not None)
    origin = first.device
    dev = first.device if first.is_cuda else cuda_device()
    out = [None if t is None else (t if t.is_cuda else t.to(dev, non_blocking=True)) for t in tensors]
    require_cuda(*out)
    return dev, origin, out


def ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def stream_ptr(device=None):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def f32c(t):
    """fp32 + contiguous view/copy of t (no copy when already so)."""
    if t.dtype != torch.float32:
        t = t.float()
    return t if t.is_contiguous() else t.contiguous()
