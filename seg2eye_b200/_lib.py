"""ctypes binding of include/seg2eye_b200.h.  There is NO fallback: if the CUDA library is missing or a
call fails, a RuntimeError is raised -- nothing on the product path routes through PyTorch library
kernels or the CPU oracle."""
import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "_C", "libseg2eye_b200.so")

MAX_TAPS = 16
ACT_NONE, ACT_LRELU, ACT_RELU = 0, 1, 2
IMPL_TC, IMPL_SIMT = 0, 1
RED_SUM, RED_HINGE_REAL, RED_HINGE_FAKE, RED_L1, RED_L2, RED_LS, RED_BCE, RED_SIGN = 0, 1, 2, 3, 4, 5, 6, 7
DIFFAUG_COLOR, DIFFAUG_TRANSLATION, DIFFAUG_CUTOUT = 1, 2, 4
DIFFAUG_XFLIP, DIFFAUG_GEOMETRIC = 8, 16
DIFFAUG_RECORD, DIFFAUG_GEOM_RECORD = 6, 8


class ConvDesc(C.Structure):
    _fields_ = [("B", C.c_int), ("Hi", C.c_int), ("Wi", C.c_int), ("Cin", C.c_int),
                ("Ho", C.c_int), ("Wo", C.c_int), ("Cout", C.c_int), ("ntaps", C.c_int),
                ("tap_dy", C.c_int * MAX_TAPS), ("tap_dx", C.c_int * MAX_TAPS), ("act", C.c_int),
                ("tile_w", C.c_int), ("tile_h", C.c_int), ("tile_b", C.c_int),
                ("ktile_w", C.c_int), ("ktile_h", C.c_int), ("ktile_b", C.c_int), ("relu_mask", C.c_void_p),
                ("residual", C.c_void_p), ("bias_n", C.c_int), ("in_act", C.c_int), ("mask_slope", C.c_float),
                ("spade_x", C.c_void_p), ("spade_par", C.c_void_p), ("spade_C", C.c_int), ("spade_act", C.c_int),
                ("spade_up", C.c_int), ("spade_gamma_out", C.c_void_p), ("spade_mask_out", C.c_void_p),
                ("spade_plain", C.c_int), ("img_out", C.c_void_p), ("img_target", C.c_void_p), ("img_sums", C.c_void_p)]


class SnJob(C.Structure):
    _fields_ = [("w", C.c_void_p), ("u", C.c_void_p), ("v", C.c_void_p), ("inv_sigma", C.c_void_p),
                ("scratch", C.c_void_p), ("u_copy", C.c_void_p), ("v_copy", C.c_void_p), ("rows", C.c_int), ("cols", C.c_int)]


class PackJob(C.Structure):
    _fields_ = [("w_oihw", C.c_void_p), ("bias", C.c_void_p), ("out_bf16", C.c_void_p), ("Cout", C.c_int), ("Cin", C.c_int), ("kh", C.c_int),
                ("kw", C.c_int), ("stride", C.c_int), ("pad", C.c_int), ("transposed", C.c_int), ("Cout_total", C.c_int),
                ("co_offset", C.c_int), ("cin_pad", C.c_int), ("im2col3x3", C.c_int)]


_P, _I, _F, _LL, _D = C.c_void_p, C.c_int, C.c_float, C.c_longlong, C.c_double
_SIGS = {
    "s2e_abi_version": [],
    "s2e_debug_set": [_I, _I],
    "s2e_onehot_nchw": [_P, _I, _I, _I, _I, _P, _P],
    "s2e_seg_nearest_nhwc": [_P, _I, _I, _I, _I, _I, _I, _I, _P, _P],
    "s2e_seg_im2col3x3": [_P, _I, _I, _I, _I, _I, _I, _P, _P],
    "s2e_pack_weight_im2col3x3": [_P, _I, _I, _P, _P],
    "s2e_unpack_wgrad_im2col3x3": [_P, _I, _I, _P, _P, _P],
    "s2e_nchw_f32_to_nhwc_bf16": [_P, _I, _I, _I, _I, _P, _P],
    "s2e_nhwc_bf16_to_nchw_f32": [_P, _I, _I, _I, _I, _P, _P],
    "s2e_tapconv_fwd": [C.POINTER(ConvDesc), _P, _P, _P, _P, _P, _I, _P],
    "s2e_tapconv_wgrad": [C.POINTER(ConvDesc), _P, _P, _P, _I, _P],
    "s2e_head_dots": [_P, _P, _LL, _I, _I, _P, _P],
    "s2e_head_gather": [C.POINTER(ConvDesc), _P, _P, _P, _P, _P, _P],
    "s2e_head_gather_signs": [C.POINTER(ConvDesc), _P, _P, _P, _P, _P, _P, _P],
    "s2e_head_scatter": [C.POINTER(ConvDesc), _P, _P, _P],
    "s2e_pack_weight": [_P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _I, _P, _P],
    "s2e_packed_taps": [_I, _I, _I, _I, C.POINTER(_I), C.POINTER(_I), C.POINTER(_I)],
    "s2e_unpack_wgrad": [_P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _P, _P, _P, _P, _P, _P, _I, _P],
    "s2e_spectral_power_iter": [_P, _I, _I, _P, _P, _P, _P, _I, _P, _P, _P],
    "s2e_spectral_power_iter_multi": [C.POINTER(SnJob), _I, _I, _I, _P],
    "s2e_pack_weight_multi": [C.POINTER(PackJob), _I, _P],
    "s2e_adam_multi": [_I, C.POINTER(_P), C.POINTER(_P), C.POINTER(_P), C.POINTER(_P), C.POINTER(_LL), _P, _F, _F, _F, _F, _P],
    "s2e_adam_multi_ema": [_I, C.POINTER(_P), C.POINTER(_P), C.POINTER(_P), C.POINTER(_P), C.POINTER(_LL), _P, _F, _F, _F, _F,
                           C.POINTER(_P), _F, _P],
    "s2e_copy_multi": [_I, C.POINTER(_P), C.POINTER(_P), C.POINTER(_LL), _P],
    "s2e_sn_in_correction": [_P, _P, _P, _I, _I, _I, _F, _P, _P, _I, _P, _P, _P],
    "s2e_space_to_depth": [_P, _I, _I, _I, _I, _P, _P],
    "s2e_depth_to_space": [_P, _I, _I, _I, _I, _P, _P],
    "s2e_norm_stats": [_P, _I, _I, _I, _I, _P, _P],
    "s2e_norm_finalize": [_P, _I, _I, _D, _D, _F, _P, _P, _P, _P, _F, _P, _P],
    "s2e_norm_merge": [_P, _I, _I, _P, _P, _P],
    "s2e_norm_finalize_merged": [_P, _P, _I, _D, _F, _P, _P, _P, _P, _F, _P, _P],
    "s2e_spade_params": [_P, _P, _P, _I, _I, _I, _P, _P],
    "s2e_spade_style_fwd": [_P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P, _P, _I, _P],
    "s2e_spade_style_bwd": [_P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P, _P, _I, _P, _P, _P, _I, _I, _P],
    "s2e_spade_style_bwd_reduce": [_P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P, _P, _P, _P, _I, _I, _P],
    "s2e_spade_style_bwd_apply": [_P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P, _P, _P, _I, _P, _I, _I, _P],
    "s2e_instnorm_fwd": [_P, _I, _I, _I, _I, _F, _P, _I, _P, _P, _P, _P, _P, _P],
    "s2e_instnorm_bwd": [_P, _P, _P, _P, _P, _I, _I, _I, _I, _P, _P, _P],
    "s2e_upsample2x_fwd": [_P, _I, _I, _I, _I, _P, _P],
    "s2e_upsample2x_bwd": [_P, _I, _I, _I, _I, _P, _P],
    "s2e_add": [_P, _P, _LL, _P, _P],
    "s2e_act_fwd": [_P, _LL, _I, _P, _P],
    "s2e_act_bwd": [_P, _P, _LL, _I, _P, _P],
    "s2e_avgpool3s2_fwd": [_P, _I, _I, _I, _I, _P, _P],
    "s2e_avgpool3s2_bwd": [_P, _I, _I, _I, _I, _P, _P],
    "s2e_bilinear_fwd": [_P, _I, _I, _I, _I, _I, _P, _P],
    "s2e_bilinear_bwd": [_P, _I, _I, _I, _I, _I, _P, _P],
    "s2e_make_d_input": [_P, _P, _P, _I, _I, _I, _I, _I, _P, _P],
    "s2e_d_input_grad": [_P, _I, _I, _I, _I, _I, _P, _P],
    "s2e_diffaug_draw": [_P, _I, _LL, _I, _I, _P, _P],
    "s2e_diffaug_means": [_P, _P, _I, _I, _I, _P, _P],
    "s2e_make_d_input_aug": [_P, _P, _P, _I, _I, _I, _I, _I, _P, _P, _I, _P, _P],
    "s2e_d_input_grad_aug": [_P, _I, _I, _I, _I, _I, _P, _I, _P, _P, _P],
    "s2e_diffaug_draw_p": [_P, _P, _I, _LL, _I, _I, _P, _P, _P],
    "s2e_make_d_input_aug_masked": [_P, _P, _P, _I, _I, _I, _I, _I, _P, _P, _I, _P, _P, _P],
    "s2e_d_input_grad_aug_masked": [_P, _I, _I, _I, _I, _I, _P, _I, _P, _P, _P, _P],
    "s2e_diffaug_draw_geom": [_P, _P, _I, _LL, _I, _I, _P, _P, _P, _P],
    "s2e_make_d_input_aug_geom": [_P, _P, _P, _I, _I, _I, _I, _I, _P, _P, _I, _P, _P, _P, _P],
    "s2e_d_input_grad_aug_geom": [_P, _I, _I, _I, _I, _I, _P, _I, _P, _P, _P, _P, _P],
    "s2e_ada_update": [_P, _I, _P, _P, _P, _D, _D, _I, _P],
    "s2e_tanh_fwd": [_P, _LL, _P, _P],
    "s2e_tanh_bwd": [_P, _P, _LL, _P, _P],
    "s2e_linear_fwd": [_P, _P, _P, _I, _I, _I, _I, _I, _P, _P],
    "s2e_linear_bwd": [_P, _P, _P, _P, _I, _I, _I, _I, _I, _P, _P, _P, _P],
    "s2e_reduce_loss": [_P, _P, _LL, _I, _I, _F, _F, _P, _I, _P],
    "s2e_reduce_loss_bwd": [_P, _P, _LL, _I, _I, _F, _F, _P, _P, _I, _P],
    "s2e_adam_prepare": [_P, _F, _F, _P],
    "s2e_adam_step": [_P, _P, _P, _P, _LL, _P, _F, _F, _F, _F, _P],
    "s2e_fill_f32": [_P, _LL, _F, _P],
    "s2e_to255_resize": [_P, _I, _I, _I, _I, _I, _I, _P, _P, _P, _P, _P],
    "s2e_openeds_score": [_P, _P, _I, _I, _I, _P, _P, _P],
    "s2e_aggregate_fwd": [_P, _I, _I, _I, _LL, _I, _P, _P, _P],
    "s2e_aggregate_bwd": [_P, _P, _I, _I, _I, _LL, _I, _P, _P],
    "s2e_label_nearest_flip": [_P, _I, _I, _I, _I, _I, _P, _P, _P],
    "s2e_pil_resample_u8": [_P, _I, _I, _I, _I, _I, _P, _P, _I, _P, _P],
    "s2e_u8_flip_normalize": [_P, _I, _I, _I, _I, _P, _P, _P],
    "s2e_u8_flip_to_i32": [_P, _I, _I, _I, _P, _P, _P],
}

_lib = None
launches = 0  # number of C-ABI compute calls issued (each issues >= 1 kernel of ours)


def exported_symbols():
    return sorted(_SIGS) + ["s2e_last_error"]


def lib():
    """Load the in-tree shared library (built by seg2eye_b200/build.py or __graft_entry__.build())."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "seg2eye_b200: CUDA library %s is missing. Build it with `python -m seg2eye_b200.build` "
                "(nvcc, sm_100a). There is no CPU / PyTorch fallback." % LIB_PATH)
        l = C.CDLL(LIB_PATH)
        l.s2e_last_error.restype = C.c_char_p
        l.s2e_last_error.argtypes = []
        for name, sig in _SIGS.items():
            fn = getattr(l, name)
            fn.restype = C.c_int
            fn.argtypes = sig
        _lib = l
        # bring-up aid: S2E_DEBUG="key=value,key=value" sets the library's debug knobs (include/seg2eye_b200.h) at load
        # time, e.g. S2E_DEBUG=5=3 runs every narrow weight gradient through the experimental multi-tap kernel
        for item in filter(None, os.environ.get("S2E_DEBUG", "").split(",")):
            k, v = item.split("=")
            if l.s2e_debug_set(int(k), int(v)) != 0:
                raise RuntimeError("S2E_DEBUG: bad debug key %s" % k)
    return _lib


def call(name, *args):
    global launches
    l = lib()
    rc = getattr(l, name)(*args)
    if rc != 0:
        raise RuntimeError("seg2eye_b200.%s failed (%d): %s" % (name, rc, l.s2e_last_error().decode()))
    launches += 1
    return rc


def ptr(t):
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("seg2eye_b200 kernels need CUDA tensors (got %s); there is no CPU fallback" % t.device)
    return t.data_ptr()


def stream():
    return torch.cuda.current_stream().cuda_stream


def packed_taps(kh, kw, stride, pad):
    n = C.c_int(0)
    dy = (C.c_int * MAX_TAPS)()
    dx = (C.c_int * MAX_TAPS)()
    l = lib()
    rc = l.s2e_packed_taps(kh, kw, stride, pad, C.byref(n), dy, dx)
    if rc != 0:
        raise RuntimeError("s2e_packed_taps failed: %s" % l.s2e_last_error().decode())
    return [(dy[i], dx[i]) for i in range(n.value)]
