"""ctypes binding of libudh.so (include/udh.h).  No CPU fallback: if the library is missing it is built with nvcc,
and if that is impossible the import fails loudly."""
import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_float, c_int, c_int64, c_size_t, c_uint32, c_uint64, c_ulonglong, c_void_p

from . import build_ext

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = build_ext.LIB

OK, EINVAL, ECUDA, ENOSUP, EWS = 0, -1, -2, -3, -4
NUMERIC_FP32, NUMERIC_BF16, NUMERIC_BF16X3 = 0, 1, 2
BWD_ALL, BWD_HEAD, BWD_CONVS = 0, 1, 2
LOSS_L1, LOSS_REC, LOSS_L1_SMOOTH, LOSS_NCC, LOSS_CUSTOM = 0, 1, 2, 3, 4
NSUMS, NLOSSES, NMETRICS = 8, 8, 4
L_REC, L_SSIM, L_L1, L_L1_SMOOTH, L_NCC = 0, 1, 2, 3, 4
M_H_LOSS, M_BOUNDED_H_LOSS, M_NUM_FAIL, M_ACE = 0, 1, 2, 3

class StepArgs(ctypes.Structure):
    """udh_step_args (include/udh.h)."""
    _fields_ = [("B", c_int), ("P", c_int), ("img_h", c_int), ("img_w", c_int), ("C", c_int),
                ("numeric_mode", c_int), ("loss_type", c_int), ("train", c_int), ("seed", c_uint64),
                ("params", c_void_p), ("grads", c_void_p), ("ws", c_void_p), ("ws_bytes", c_size_t),
                ("I1", c_void_p), ("I2", c_void_p), ("I_aug", c_void_p), ("pts1", c_void_p), ("gt", c_void_p),
                ("patch_indices", c_void_p), ("idx_stride", c_int64),
                ("h4p", c_void_p), ("H", c_void_p), ("pred_I2", c_void_p),
                ("dh4p", c_void_p), ("dH", c_void_p), ("scratch", c_void_p), ("dpred_map", c_void_p), ("sums", c_void_p),
                ("photo_losses", c_void_p), ("h4p_metrics", c_void_p), ("per_sample", c_void_p), ("fwd_flags", c_int)]


FWD_FC1_MIRROR_CURRENT = 1


STEP_ALL, STEP_FWD_HEAD, STEP_CONVS, STEP_FWD_ONLY = 0, 1, 2, 3
STEP_LOSS = {"h_loss": 0, "l1_loss": 1, "rec_loss": 2, "l1_smooth_loss": 3, "ncc_loss": 4, "ssim_loss": 5}


# name -> (restype, argtypes); every symbol include/udh.h declares
SIGNATURES = {
    "udh_version": (c_int, []),
    "udh_last_error": (c_char_p, []),
    "udh_device_available": (c_int, []),
    "udh_dlt_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    "udh_dlt_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    "udh_warp_loss_fwd": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_int,
                                  c_void_p, c_void_p, c_int, c_void_p]),
    "udh_warp_loss_fwd_ex": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_int,
                                     c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "udh_warp_loss_bwd": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_int, c_int,
                                  c_void_p, c_float, c_void_p, c_void_p, c_int, c_void_p]),
    "udh_warp_loss_bwd_ex": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_int, c_int,
                                     c_void_p, c_void_p, c_float, c_void_p, c_void_p, c_int, c_void_p]),
    "udh_ssim_bwd": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_int, c_void_p]),
    "udh_ssim_fwd": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_int, c_void_p]),
    "udh_photo_losses_finalize": (c_int, [c_void_p, c_double, c_double, c_void_p, c_void_p]),
    "udh_transformer_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "udh_h4p_loss": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "udh_cnn_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "udh_cnn_workspace_init": (c_int, [c_void_p, c_size_t, c_int, c_int, c_int, c_void_p]),
    "udh_cnn_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_int, c_int, c_int, c_uint64, c_int,
                            c_void_p]),
    "udh_cnn_fwd_ex": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_int, c_int, c_int, c_uint64, c_int,
                               c_int, c_void_p]),
    "udh_cnn_fc1_mirror": (c_int, [c_void_p, c_size_t, c_int, c_int, c_int, POINTER(c_void_p), POINTER(c_size_t), POINTER(c_size_t),
                                   POINTER(c_int)]),
    "udh_cnn_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_int, c_int, c_int, c_int,
                            c_void_p]),
    "udh_cnn_bwd_phase": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_int, c_int, c_int, c_int,
                                  c_int, c_void_p]),
    "udh_cnn_dropout_masks": (c_int, [c_void_p, c_size_t, c_int, c_int, c_int, POINTER(c_void_p), POINTER(c_void_p)]),
    "udh_cnn_activation": (c_int, [c_void_p, c_size_t, c_int, c_int, c_int, c_int, POINTER(c_void_p), POINTER(c_size_t)]),
    "udh_param_offset": (c_int, [c_int, c_int, POINTER(c_size_t), POINTER(c_size_t)]),
    "udh_param_total_floats": (c_size_t, [c_int]),
    "udh_adam_step": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_float, c_float, c_float, c_float, c_float,
                              c_int, c_void_p]),
    "udh_adam_step_mirror": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_float, c_float, c_float, c_float, c_float,
                                     c_int, c_void_p, c_size_t, c_size_t, c_int, c_void_p]),
    "udh_adam_step_mirror_ex": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_float, c_float, c_float, c_float, c_float,
                                        c_int, c_void_p, c_size_t, c_size_t, c_int, c_int, c_void_p]),
    "udh_dp_shard_update": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_size_t, c_size_t, c_size_t,
                                    c_int, c_float, c_float, c_float, c_float, c_float, c_int, c_void_p]),
    "udh_debug_x3_materialize": (c_int, [c_void_p, c_size_t, c_int, c_int, POINTER(c_size_t), c_void_p]),
    "udh_debug_x3_set_rows": (c_int, [c_int]),
    "udh_debug_x3_scratch_bytes": (c_size_t, [c_int, c_int, c_int, c_int, c_int]),
    "udh_debug_x3_conv": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                                  c_void_p]),
    "udh_debug_x3_wgrad": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "udh_debug_x3_conv1": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int,
                                   c_int, c_void_p]),
    "udh_debug_tc_conv_scratch_bytes": (c_size_t, [c_int, c_int, c_int, c_int, c_int]),
    "udh_debug_tc_conv": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                          c_void_p]),
    "udh_debug_tc_conv_pool": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "udh_debug_tc_wgrad": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "udh_step_forward_backward": (c_int, [POINTER(StepArgs), c_int, c_void_p]),
    "udh_prep_inputs_u8": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                                   c_void_p]),
    "udh_prep_inputs_u8_ex": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                      c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "udh_synth_scene_u8": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_uint64, c_void_p]),
    "udh_warp_image_u8": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "udh_launch_count": (c_ulonglong, []),
    "udh_set_sm_reserve_top": (c_int, [c_int]),
    "udh_crc32c": (c_uint32, [c_void_p, c_size_t, c_uint32]),
    "udh_set_bwd_marker": (c_int, [c_int]),
    "udh_bwd_marker_wait": (c_int, [c_void_p]),
    "udh_prof_enable": (c_int, [c_int]),
    "udh_prof_reset": (c_int, []),
    "udh_prof_num_tags": (c_int, []),
    "udh_prof_tag_name": (c_char_p, [c_int]),
    "udh_prof_read": (c_int, [c_int, POINTER(c_float), POINTER(c_int)]),
}


class UdhError(RuntimeError):
    pass


def _load():
    if build_ext.needs_build():
        build_ext.build()      # raises if nvcc is unavailable: there is deliberately no pure-Python/CPU path
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    return lib


lib = _load()


def check(rc, what=""):
    if rc != OK:
        raise UdhError("%s failed (%d): %s" % (what or "libudh call", rc, lib.udh_last_error().decode()))


def require_device():
    if not lib.udh_device_available():
        raise UdhError("no CUDA device: libudh has no CPU fallback (the CPU oracle lives in oracle/ and is test-only)")


def prof_read_all():
    """{tag name: (total_ms, count)} of the library's per-phase CUDA-event timers (non-empty phases only)."""
    out = {}
    for t in range(lib.udh_prof_num_tags()):
        ms, n = c_float(), c_int()
        check(lib.udh_prof_read(t, ctypes.byref(ms), ctypes.byref(n)), "udh_prof_read")
        if n.value:
            out[lib.udh_prof_tag_name(t).decode()] = (ms.value, n.value)
    return out


def load_probes():
    """libudh_probe.so (include/udh_probe.h): hardware probes, built on demand, never loaded by the product path."""
    plib = ctypes.CDLL(build_ext.build_probes())
    plib.udh_debug_umma_probe.restype = c_int
    plib.udh_debug_umma_probe.argtypes = [c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_int, c_void_p]
    plib.udh_debug_umma2_probe.restype = c_int
    plib.udh_debug_umma2_probe.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]
    return plib
