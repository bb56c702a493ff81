"""ctypes binding of libcrfr.so (the C-ABI declared in include/crfr.h).

There is no CPU fallback: if the library is missing or a call fails, a RuntimeError is raised.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libcrfr.so")

ENGINE_AUTO, ENGINE_DIRECT, ENGINE_TCGEN05 = 0, 1, 2
FSRNET_NPARAMS = 202

vp, ci, cf, cll, csz = C.c_void_p, C.c_int, C.c_float, C.c_longlong, C.c_size_t


class ConvDesc(C.Structure):
    _fields_ = [(k, ci) for k in ("n", "h", "w", "cin", "cout", "k", "stride", "pad", "oh", "ow", "in_ld", "out_ld",
                                  "transposed")]


class FsrnetIO(C.Structure):
    _fields_ = [("batch", ci), ("size", ci), ("x", vp), ("coarse", vp), ("out", vp), ("landmark", vp), ("parsing", vp),
                ("hr", vp), ("heatmap", vp), ("labels", vp), ("loss_div", cf), ("w_pix", cf), ("bucket_events", vp * 3)]


class FsrnetIdIO(C.Structure):
    _fields_ = [("teacher_layers", ci), ("teacher_se", ci), ("teacher_params", vp), ("teacher_buffers", vp), ("w_id", cf),
                ("terms", ci), ("id_scale", cf)]


class TapeEntry(C.Structure):
    _fields_ = [("kind", ci), ("n", ci), ("h", ci), ("w", ci), ("c", ci), ("ld", ci), ("out_off", cll),
                ("in_off", cll), ("stats_off", cll), ("w_idx", ci), ("has_res", ci)]


class FsrnetSectionIO(C.Structure):
    _fields_ = [("section", ci), ("batch", ci), ("size", ci), ("x", vp), ("out", vp * 3)]


FSRNET_COARSE, FSRNET_ENCODER, FSRNET_PRIOR, FSRNET_DECODER = 0, 1, 2, 3


class SrnetIO(C.Structure):
    _fields_ = [("section", ci), ("batch", ci), ("h", ci), ("w", ci), ("x", vp), ("out", vp * 4)]


# SUPER_RESOLUTION FSRNet variant program (crfr_srnet_*): sections and their state_dict lengths
SRNET_COARSE, SRNET_ENCODER, SRNET_PRIOR, SRNET_DECODER, SRNET_NETWORK = 0, 1, 2, 3, 4
SRNET_NPARAMS = {SRNET_COARSE: 52, SRNET_ENCODER: 51, SRNET_PRIOR: 954, SRNET_DECODER: 51, SRNET_NETWORK: 1108}


class ResnetIO(C.Structure):
    _fields_ = [("batch", ci), ("size", ci), ("x", vp), ("emb", vp), ("feat", vp * 4), ("training", ci),
                ("momentum", cf), ("eps", cf)]


class KdIO(C.Structure):
    _fields_ = [("batch", ci), ("size", ci), ("x", vp), ("momentum", cf), ("eps", cf), ("assistant_grad_to_student", ci),
                ("x_lr", vp), ("teacher_ir50", ci), ("events", vp * 2), ("teacher_ir_layers", ci), ("teacher_ir_se", ci)]


RESNET34_NPARAMS, RESNET34_NBN = 114, 38
IR50_NPARAMS, IR50_NBN = 187, 54

# name -> (restype, argtypes); every symbol declared in include/crfr.h
SIGNATURES = {
    "crfr_last_error": (C.c_char_p, []),
    "crfr_version": (ci, []),
    "crfr_launch_count": (C.c_ulonglong, []),
    "crfr_set_option": (ci, [C.c_char_p, ci]),
    "crfr_conv_engine_supported": (ci, [ci] * 9),
    "crfr_nchw_f32_to_nhwc_bf16": (ci, [vp, vp, ci, ci, ci, ci, ci, ci, vp]),
    "crfr_nhwc_bf16_to_nchw_f32": (ci, [vp, vp, ci, ci, ci, ci, ci, vp]),
    "crfr_pack_weight": (ci, [vp, vp, ci, ci, ci, ci, cll, cll, cll, vp]),
    "crfr_conv_fwd": (ci, [ci, C.POINTER(ConvDesc), vp, vp, ci, vp, vp, vp, vp, cf, vp, csz, vp]),
    "crfr_conv_dgrad": (ci, [ci, C.POINTER(ConvDesc), vp, vp, ci, vp, vp, csz, vp]),
    "crfr_conv_wgrad": (ci, [ci, C.POINTER(ConvDesc), vp, vp, vp, vp, vp, csz, vp]),
    "crfr_conv_workspace_bytes": (csz, [C.POINTER(ConvDesc)]),
    "crfr_norm_workspace_bytes": (csz, [ci, ci, ci]),
    "crfr_norm_stats": (ci, [vp, ci, ci, ci, ci, cf, vp, vp, csz, vp]),
    "crfr_norm_act_fwd": (ci, [vp, ci, vp, vp, vp, vp, ci, vp, ci, vp, ci, ci, ci, ci, vp]),
    "crfr_norm_act_bwd": (ci, [vp, ci, vp, ci, vp, ci, vp, vp, vp, vp, ci, vp, ci, vp, ci, vp, ci, vp, vp, vp, ci, ci,
                               ci, vp, csz, vp]),
    "crfr_conv_dgrad_norm_bwd_workspace_bytes": (csz, [C.POINTER(ConvDesc)]),
    "crfr_conv_dgrad_norm_bwd": (ci, [ci, C.POINTER(ConvDesc), vp, vp, ci, vp, ci, vp, ci, vp, vp, vp, vp, ci, vp, ci, vp,
                                      ci, vp, ci, vp, vp, vp, vp, csz, vp]),
    "crfr_maxpool2_fwd": (ci, [vp, ci, vp, ci, ci, ci, ci, ci, vp]),
    "crfr_maxpool2_bwd": (ci, [vp, ci, vp, ci, vp, ci, ci, ci, ci, ci, vp]),
    "crfr_upnearest2_add_fwd": (ci, [vp, ci, vp, ci, vp, ci, ci, ci, ci, ci, vp]),
    "crfr_upnearest2_bwd": (ci, [vp, ci, vp, ci, ci, ci, ci, ci, vp]),
    "crfr_add_n": (ci, [vp, ci, vp, ci, vp, ci, vp, ci, cll, ci, vp]),
    "crfr_loss_mse97": (ci, [vp, vp, ci, ci, ci, cf, vp, vp, ci, vp, csz, vp]),
    "crfr_loss_landmark": (ci, [vp, vp, ci, ci, ci, cf, vp, vp, ci, ci, vp, csz, vp]),
    "crfr_loss_ce2d": (ci, [vp, vp, ci, ci, ci, cf, vp, vp, ci, ci, vp, csz, vp]),
    "crfr_loss_kd": (ci, [vp, vp, vp, cll, ci, cf, vp, vp, vp, vp, vp, csz, vp]),
    "crfr_rmsprop_step": (ci, [vp, vp, vp, cll, cf, cf, cf, cf, cf, vp]),
    "crfr_bicubic_table_size": (ci, [ci, ci]),
    "crfr_bicubic_tables": (ci, [ci, ci, vp]),
    "crfr_bicubic_u8": (ci, [vp, ci, ci, ci, ci, vp, vp, ci, ci, vp, vp, vp, vp]),
    "crfr_landmark_heatmap": (ci, [vp, ci, ci, cf, ci, ci, vp, vp]),
    "crfr_rotate_coeffs": (ci, [ci, ci, C.c_double, vp]),
    "crfr_augment_u8": (ci, [vp, ci, ci, ci, ci, vp, vp, ci, vp, vp]),
    "crfr_crop_u8": (ci, [vp, ci, ci, ci, ci, vp, ci, ci, vp, vp]),
    "crfr_l2norm_bf16": (ci, [vp, vp, cll, ci, vp]),
    "crfr_cosine_topk": (ci, [ci, vp, vp, ci, cll, ci, ci, ci, vp, vp, vp, csz, vp]),
    "crfr_cosine_topk_workspace_bytes": (csz, [ci, cll, ci, ci]),
    "crfr_topk_merge": (ci, [vp, vp, ci, ci, ci, vp, vp, vp]),
    "crfr_topk_rows": (ci, [vp, ci, cll, ci, vp, vp, vp]),
    "crfr_verify_counts": (ci, [vp, vp, cll, cf, vp, vp]),
    "crfr_verify_sweep": (ci, [vp, vp, vp, ci, vp, ci, vp, vp]),
    "crfr_pair_verify": (ci, [vp, vp, cll, ci, cf, vp, vp, vp]),
    "crfr_reflect_pad_fwd": (ci, [vp, ci, vp, ci, ci, ci, ci, ci, ci, vp]),
    "crfr_reflect_pad_bwd": (ci, [vp, ci, vp, ci, ci, ci, ci, ci, ci, vp]),
    "crfr_tanh_fwd": (ci, [vp, vp, cll, vp]),
    "crfr_tanh_bwd": (ci, [vp, vp, vp, cll, vp]),
    "crfr_linear_workspace_bytes": (csz, [ci, ci, ci, ci]),
    "crfr_linear_fwd": (ci, [vp, ci, ci, ci, vp, vp, ci, vp, vp, csz, vp]),
    "crfr_linear_bwd": (ci, [vp, vp, ci, ci, ci, vp, ci, vp, vp, vp, vp, csz, vp]),
    "crfr_fsrnet_workspace_bytes": (csz, [ci, ci, ci]),
    "crfr_fsrnet_tape": (ci, [ci, ci, ci, C.POINTER(TapeEntry), ci]),
    "crfr_fsrnet_id_tape": (ci, [ci, ci, ci, ci, ci, C.POINTER(TapeEntry), ci]),
    "crfr_fsrnet_forward": (ci, [ci, vp, C.POINTER(FsrnetIO), ci, vp, csz, vp]),
    "crfr_fsrnet_backward": (ci, [ci, vp, vp, C.POINTER(FsrnetIO), vp, vp, vp, vp, vp, csz, vp]),
    "crfr_fsrnet_section_workspace_bytes": (csz, [ci, ci, ci, ci]),
    "crfr_fsrnet_section_forward": (ci, [ci, vp, C.POINTER(FsrnetSectionIO), ci, vp, csz, vp]),
    "crfr_fsrnet_section_backward": (ci, [ci, vp, vp, C.POINTER(FsrnetSectionIO), vp, vp, vp, csz, vp]),
    "crfr_fsrnet_train_step": (ci, [ci, vp, vp, C.POINTER(FsrnetIO), vp, vp, csz, vp]),
    "crfr_fsrnet_id_workspace_bytes": (csz, [ci, ci, ci, ci]),
    "crfr_fsrnet_id_train_step": (ci, [ci, vp, vp, C.POINTER(FsrnetIO), C.POINTER(FsrnetIdIO), vp, vp, csz, vp]),
    "crfr_srnet_workspace_bytes": (csz, [ci, ci, ci, ci, ci]),
    "crfr_srnet_tape": (ci, [ci, ci, ci, ci, ci, C.POINTER(TapeEntry), ci]),
    "crfr_srnet_grad_tape": (ci, [ci, ci, ci, ci, ci, ci, C.POINTER(TapeEntry), ci]),
    "crfr_srnet_forward": (ci, [ci, vp, C.POINTER(SrnetIO), ci, vp, csz, vp]),
    "crfr_srnet_backward": (ci, [ci, vp, vp, C.POINTER(SrnetIO), vp, vp, vp, csz, vp]),
    "crfr_bn_update_running": (ci, [vp, vp, vp, vp, ci, cll, cf, cf, vp]),
    "crfr_bn_running_to_stats": (ci, [vp, vp, ci, cf, vp, vp]),
    "crfr_resnet34_workspace_bytes": (csz, [ci, ci, ci]),
    "crfr_resnet34_tape": (ci, [ci, ci, ci, C.POINTER(TapeEntry), ci]),
    "crfr_resnet34_forward": (ci, [ci, vp, vp, C.POINTER(ResnetIO), vp, csz, vp]),
    "crfr_kd_workspace_bytes": (csz, [ci, ci]),
    "crfr_kd_workspace_bytes_ex": (csz, [ci, ci, ci]),
    "crfr_kd_train_step": (ci, [ci, vp, vp, vp, vp, vp, vp, vp, vp, C.POINTER(KdIO), vp, vp, csz, vp]),
    "crfr_ir50_workspace_bytes": (csz, [ci, ci]),
    "crfr_ir50_forward": (ci, [ci, vp, vp, C.POINTER(ResnetIO), vp, csz, vp]),
    "crfr_ir50_grad_workspace_bytes": (csz, [ci, ci]),
    "crfr_ir50_tape": (ci, [ci, ci, C.POINTER(TapeEntry), ci]),
    "crfr_ir50_backward": (ci, [ci, vp, vp, C.POINTER(ResnetIO), vp, vp, vp, vp, csz, vp]),
    "crfr_resnet34_backward": (ci, [ci, vp, vp, C.POINTER(ResnetIO), vp, vp, vp, csz, vp]),
    "crfr_kd_workspace_bytes_ir": (csz, [ci, ci, ci, ci]),
    "crfr_irnet_sizes": (ci, [ci, ci, C.POINTER(ci), C.POINTER(ci)]),
    "crfr_irnet_workspace_bytes": (csz, [ci, ci, ci, ci]),
    "crfr_irnet_forward": (ci, [ci, ci, ci, vp, vp, C.POINTER(ResnetIO), vp, csz, vp]),
    "crfr_irnet_grad_workspace_bytes": (csz, [ci, ci, ci, ci]),
    "crfr_irnet_tape": (ci, [ci, ci, ci, ci, C.POINTER(TapeEntry), ci]),
    "crfr_irnet_grad_tape": (ci, [ci, ci, ci, ci, ci, C.POINTER(TapeEntry), ci]),
    "crfr_irnet_backward": (ci, [ci, ci, ci, vp, vp, C.POINTER(ResnetIO), vp, vp, vp, vp, csz, vp]),
}

_lib = None


def lib():
    """Loads libcrfr.so (once).  Raises if it has not been built: the product path has no fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError("libcrfr.so is missing (%s): run `python __graft_entry__.py` / crfr_b200.build()"
                               % LIB_PATH)
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(l, name)
            fn.restype, fn.argtypes = res, args
        _lib = l
    return _lib


def check(rc, what=""):
    if rc != 0:
        msg = lib().crfr_last_error().decode("utf-8", "replace")
        raise RuntimeError("libcrfr %s failed (code %d): %s" % (what, rc, msg))


def call(name, *args):
    check(getattr(lib(), name)(*args), name)


def irnet_sizes(num_layers, se):
    """(named_parameters count, BatchNorm count) of the IR variant (num_layers, se) (crfr_irnet_sizes)."""
    n_params, n_bn = ci(), ci()
    call("crfr_irnet_sizes", num_layers, int(se), C.byref(n_params), C.byref(n_bn))
    return n_params.value, n_bn.value
