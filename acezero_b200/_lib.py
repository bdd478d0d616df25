"""ctypes binding of libacez.so (the C ABI declared in include/acez.h).

There is no fallback: if the shared library is missing or a call fails, an exception is raised.
"""
import ctypes as C
import os
from pathlib import Path

_HERE = Path(__file__).resolve().parent
LIB_PATH = _HERE / "libacez.so"


class AcezError(RuntimeError):
    pass


class GemmDesc(C.Structure):
    _fields_ = [
        ("A", C.c_void_p), ("B", C.c_void_p),
        ("a_mn_major", C.c_int), ("b_mn_major", C.c_int),
        ("M", C.c_int), ("N", C.c_int), ("K", C.c_int), ("batch", C.c_int),
        ("a_zstride", C.c_longlong), ("b_zstride", C.c_longlong),
        ("lda", C.c_int), ("ldb", C.c_int),
        ("bn", C.c_int), ("epilogue", C.c_int),
        ("bias", C.c_void_p), ("resid", C.c_void_p), ("mask", C.c_void_p), ("addend", C.c_void_p),
        ("out", C.c_void_p), ("out2", C.c_void_p),
        ("ldo", C.c_int), ("relu", C.c_int),
        ("nonfinite", C.c_void_p),
        ("out32", C.c_void_p), ("out32_zstride", C.c_longlong), ("ldo32", C.c_int),
        ("bias_grad", C.c_void_p), ("bias_grad_zstride", C.c_longlong),
        ("a_lbo", C.c_uint), ("a_sbo", C.c_uint), ("a_kstep", C.c_uint),
        ("b_lbo", C.c_uint), ("b_sbo", C.c_uint), ("b_kstep", C.c_uint),
        ("dbg_clock", C.c_void_p),
    ]


class LossParams(C.Structure):
    _fields_ = [
        ("loss_type", C.c_int), ("loss_weight", C.c_float),
        ("depth_min", C.c_float), ("depth_max", C.c_float), ("hard_clamp", C.c_float),
        ("inlier_px", C.c_float), ("depth_target", C.c_float),
        ("use_depth", C.c_int), ("grad_scale", C.c_float), ("divisor", C.c_int),
    ]


class HeadConfig(C.Structure):
    _fields_ = [
        ("num_res_blocks", C.c_int), ("use_homogeneous", C.c_int), ("max_rows", C.c_int), ("training", C.c_int),
        ("mean", C.c_float * 3),
        ("h_beta", C.c_float), ("max_inv_scale", C.c_float), ("min_inv_scale", C.c_float),
    ]


class TrainBatch(C.Structure):
    _fields_ = [
        ("features", C.c_void_p), ("target_px_b2", C.c_void_p), ("P_b34", C.c_void_p),
        ("aug_inv_b34", C.c_void_p), ("pose_inv_b44", C.c_void_p), ("K_b33", C.c_void_p), ("Kinv_b33", C.c_void_p),
        ("target_crds_b3", C.c_void_p), ("d_P_b34", C.c_void_p), ("d_Kdiag_b2", C.c_void_p),
        ("sc_out_b3", C.c_void_p), ("grad_scale_dev", C.c_void_p), ("loss_weight_dev", C.c_void_p),
    ]


class DsacParams(C.Structure):
    _fields_ = [
        ("hyps", C.c_int), ("inlier_threshold", C.c_float), ("inlier_alpha", C.c_float), ("max_reproj", C.c_float),
        ("subsample", C.c_int), ("seed", C.c_uint64), ("max_tries", C.c_int), ("max_refine_steps", C.c_int),
        ("image_index_base", C.c_int), ("image_index", C.c_void_p),
    ]


class ScheduleParams(C.Structure):
    _fields_ = [
        ("kind", C.c_int), ("iterations", C.c_int), ("lr_min", C.c_float), ("lr_max", C.c_float),
        ("warmup_iterations", C.c_int), ("warmup_lr", C.c_float), ("cooldown_iterations", C.c_int),
        ("cooldown_trigger", C.c_float), ("batch_global", C.c_int), ("loss_dyntanh", C.c_int),
        ("loss_schedule_circle", C.c_int), ("soft_clamp", C.c_float), ("soft_clamp_min", C.c_float),
    ]


SCHED_STATE_FLOATS = 128
SCHED_KINDS = {"constant": 0, "circle": 1, "1cyclepoly": 2}


class ImagePrepDesc(C.Structure):
    _fields_ = [
        ("src", C.c_void_p), ("h_in", C.c_int), ("w_in", C.c_int), ("channels", C.c_int),
        ("coef_x", C.c_void_p), ("coef_y", C.c_void_p), ("kx", C.c_int), ("ky", C.c_int),
        ("contrast_first", C.c_int), ("brightness", C.c_float), ("contrast", C.c_float), ("rotate", C.c_int),
        ("affine", C.c_double * 6),
    ]


class DsacDebug(C.Structure):
    _fields_ = [
        ("hyp_poses", C.c_void_p), ("hyp_scores", C.c_void_p), ("best", C.c_void_p), ("hyp_tries", C.c_void_p),
        ("refine_rounds", C.c_void_p),
    ]


_lib = None

# every symbol include/acez.h declares (the CPU test checks the .so exports all of them)
EXPORTS = [
    "acez_version", "acez_last_error", "acez_device_check", "acez_gemm_f16", "acez_repro_loss_fwd_bwd",
    "acez_head_param_count", "acez_head_workspace_bytes", "acez_head_plan_create", "acez_head_plan_destroy",
    "acez_head_sync_weights", "acez_head_input_ptr", "acez_head_plan_fused_chain", "acez_debug_chain_clocks", "acez_head_forward", "acez_head_forward_train",
    "acez_head_backward", "acez_head_train_fwd_bwd",
    "acez_adamw_dp_shard", "acez_adamw_dp_step", "acez_head_w16_ptr", "acez_gather_rows", "acez_gather_rows_multi", "acez_buffer_fill", "acez_adamw_step", "acez_schedule_init", "acez_schedule_step", "acez_gather_rows_multi_sched", "acez_dsac_workspace_bytes", "acez_dsac_forward_rgb_batch",
    "acez_encoder_workspace_bytes", "acez_encoder_plan_create", "acez_encoder_plan_destroy", "acez_encoder_out_hw",
    "acez_encoder_forward", "acez_pointcloud_metrics",
    "acez_image_prep_workspace_bytes", "acez_image_prep", "acez_image_mask_cells",
]


def load():
    """Load libacez.so; raises AcezError when it has not been built (no silent fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise AcezError(f"{LIB_PATH} not found: build it with `python -m acezero_b200.build` "
                        "(acezero_b200 has no CPU or PyTorch fallback path)")
    lib = C.CDLL(str(LIB_PATH))
    lib.acez_last_error.restype = C.c_char_p
    lib.acez_version.restype = C.c_int
    vp, i, f = C.c_void_p, C.c_int, C.c_float
    lib.acez_gemm_f16.argtypes = [C.POINTER(GemmDesc), vp]
    lib.acez_repro_loss_fwd_bwd.argtypes = [C.POINTER(LossParams), i] + [vp] * 13
    lib.acez_head_param_count.argtypes = [C.POINTER(HeadConfig)]
    lib.acez_head_param_count.restype = C.c_size_t
    lib.acez_head_workspace_bytes.argtypes = [C.POINTER(HeadConfig)]
    lib.acez_head_workspace_bytes.restype = C.c_size_t
    lib.acez_head_plan_create.argtypes = [C.POINTER(HeadConfig), vp, vp, vp, C.c_size_t, C.POINTER(vp)]
    lib.acez_head_plan_destroy.argtypes = [vp]
    lib.acez_head_plan_destroy.restype = None
    lib.acez_head_sync_weights.argtypes = [vp, vp]
    lib.acez_head_w16_ptr.argtypes = [vp, i]
    lib.acez_head_w16_ptr.restype = vp
    lib.acez_adamw_dp_shard.argtypes = [C.c_size_t, i]
    lib.acez_adamw_dp_shard.restype = C.c_size_t
    lib.acez_adamw_dp_step.argtypes = [vp, vp, vp, vp, vp, i, i, C.c_size_t, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, i, i, vp]
    lib.acez_head_input_ptr.argtypes = [vp]
    lib.acez_head_input_ptr.restype = vp
    lib.acez_head_plan_fused_chain.argtypes = [vp]
    lib.acez_debug_chain_clocks.argtypes = [vp, C.c_size_t, C.POINTER(i)]
    lib.acez_head_forward.argtypes = [vp, vp, i, vp, vp]
    lib.acez_head_forward_train.argtypes = [vp, vp, i, vp, vp]
    lib.acez_head_backward.argtypes = [vp, i, vp, vp, vp]
    lib.acez_head_train_fwd_bwd.argtypes = [vp, i, C.POINTER(LossParams), C.POINTER(TrainBatch), vp, vp, vp]
    lib.acez_gather_rows.argtypes = [vp, vp, i, i, vp, vp]
    lib.acez_gather_rows_multi.argtypes = [vp, vp, vp, i, vp, i, vp]
    lib.acez_buffer_fill.argtypes = [vp, vp, i, i, i, i, vp, vp, i, C.c_longlong] + [vp] * 8 + [vp]
    lib.acez_adamw_step.argtypes = [vp, vp, vp, vp, C.c_size_t, vp, vp, vp, i, vp, vp]
    lib.acez_schedule_init.argtypes = [C.POINTER(ScheduleParams), vp, vp]
    lib.acez_schedule_step.argtypes = [C.POINTER(ScheduleParams), vp, vp, vp, vp]
    lib.acez_gather_rows_multi_sched.argtypes = [vp, vp, vp, i, vp, i, C.POINTER(ScheduleParams), vp, vp, vp, vp]
    lib.acez_dsac_workspace_bytes.argtypes = [i, i, i, i]
    lib.acez_dsac_workspace_bytes.restype = C.c_size_t
    lib.acez_dsac_forward_rgb_batch.argtypes = [vp, i, i, i, vp, vp, vp, C.POINTER(DsacParams), vp, vp, vp,
                                                C.POINTER(DsacDebug), vp, C.c_size_t, vp]
    lib.acez_encoder_workspace_bytes.argtypes = [i, i, i]
    lib.acez_encoder_workspace_bytes.restype = C.c_size_t
    lib.acez_encoder_plan_create.argtypes = [C.POINTER(vp), i, i, i, vp, C.c_size_t, vp, C.POINTER(vp)]
    lib.acez_encoder_plan_destroy.argtypes = [vp]
    lib.acez_encoder_plan_destroy.restype = None
    lib.acez_encoder_out_hw.argtypes = [i, i, C.POINTER(i), C.POINTER(i)]
    lib.acez_encoder_forward.argtypes = [vp, vp, i, i, i, i, vp, vp]
    lib.acez_pointcloud_metrics.argtypes = [vp, i, i, i, vp, vp, i, vp, vp, vp, vp]
    lib.acez_image_prep_workspace_bytes.argtypes = [C.POINTER(ImagePrepDesc), i, i, i]
    lib.acez_image_prep_workspace_bytes.restype = C.c_size_t
    lib.acez_image_prep.argtypes = [C.POINTER(ImagePrepDesc), i, i, i, vp, C.c_size_t, vp, vp]
    lib.acez_image_mask_cells.argtypes = [C.POINTER(C.c_double), i, i, i, i, vp, vp]
    lib.acez_host_resize_sample.argtypes = [vp, C.c_longlong, vp, i]
    lib.acez_host_jitter.argtypes = [i, i, f, f, i]
    lib.acez_host_normalize.restype = f
    lib.acez_host_rotate_sample.argtypes = [C.POINTER(C.c_double), vp, i, i, i, i]
    lib.acez_host_rotate_sample.restype = C.c_double
    lib.acez_host_mask_cell.argtypes = [C.POINTER(C.c_double), i, i, i, i, i, i]
    _lib = lib
    return lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = load().acez_last_error().decode("utf-8", "replace")
        raise AcezError(f"{what} failed (status {rc}): {msg}")


def ptr(t):
    """Device/host pointer of a torch tensor (or None)."""
    if t is None:
        return None
    return C.c_void_p(t.data_ptr())


def stream_ptr(stream=None):
    import torch
    s = stream if stream is not None else torch.cuda.current_stream()
    return C.c_void_p(s.cuda_stream)
