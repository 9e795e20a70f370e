"""ctypes binding of ``libsci_b200.so`` (C ABI declared in ``include/sci_b200.h``).

There is NO fallback: if the shared library is missing the import fails loudly
(build it with ``python adaptivepnp_sci_b200/csrc/build.py`` or
``__graft_entry__.build()``), and every entry point raises ``SciError`` on a
non-zero return code.  Tensors stay owned by PyTorch; the binding passes
``data_ptr()`` and the current CUDA stream.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libsci_b200.so")

if not os.path.exists(LIB_PATH):
    raise ImportError(
        "adaptivepnp_sci_b200: %s not found. The product has no CPU/PyTorch fallback; build the sm_100a "
        "library first: python adaptivepnp_sci_b200/csrc/build.py" % LIB_PATH)

lib = ctypes.CDLL(LIB_PATH)

_p = ctypes.c_void_p
_i = ctypes.c_int
_l = ctypes.c_long
_f = ctypes.c_float
_sz = ctypes.c_size_t
_d = ctypes.c_double

# name -> argtypes (restype int unless noted).  tests/test_capi_symbols.py checks this table against
# include/sci_b200.h so a symbol cannot be declared without being bound, or bound without being declared.
PROTOTYPES = {
    "sci_version": [],
    "sci_pixlast_to_planar": [_p, _p, _i, _i, _i, _p],
    "sci_planar_to_pixlast": [_p, _p, _i, _i, _i, _p],
    "sci_bayer_split_init": [_p, _p, _p, _p, _p, _p, _i, _i, _i, _p],
    "sci_A": [_p, _l, _l, _l, _p, _l, _l, _l, _p, _l, _l, _i, _i, _i, _p],
    "sci_At": [_p, _l, _l, _p, _l, _l, _l, _p, _l, _l, _l, _i, _i, _i, _p],
    "sci_project_stage1": [_p, _p, _p, _p, _p, _p, _l, _i, _f, _f, _p, _p, _p],
    "sci_project_stage2": [_p, _p, _p, _p, _p, _p, _l, _i, _d, _d, _p],
    "sci_tv_chambolle2d": [_p, _p, _f, _p, _p, _f, _i, _i, _i, _i, _f, _f, _i, _p, _sz, _p, _p],
    "sci_tv_strip_main": [_p, _p, _f, _p, _p, _f, _i, _i, _i, _i, _i, _i, _p, _p, _p, _p, ctypes.c_uint, _p, _f, _f, _i,
                          _p, _sz, _p, _p],
    "sci_tv_strip_finish": [_p, _p, _f, _p, _p, _f, _i, _i, _i, _i, _i, _i, _p, _p, _f, _f, _i, _p, _sz, _p, _i, _p, _p],
    "sci_malvar2004": [_p, _p, _f, _p, _f, _p, _p, _i, _i, _i, _p],
    "sci_dual_update_rgb": [_p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _p, _p, _p],
    "sci_dual_update_stage1": [_p, _p, _p, _p, _i, _i, _i, _i, _p, _p, _p],
    "sci_reflect_pad2d": [_p, _p, _l, _i, _i, _i, _i, _p],
    "sci_replicate_pad2d": [_p, _p, _l, _i, _i, _i, _i, _p],
    "sci_crop2d": [_p, _p, _l, _i, _i, _i, _i, _p],
    "sci_closed_form_demosaic": [_p, _p, _p, _p, _f, _f, _f, _i, _p, _p, _i, _i, _i, _p],
    "sci_rgb_to_bayer": [_p, _p, _i, _i, _i, _p],
    "sci_bayer_to_rgb_sparse": [_p, _p, _i, _i, _i, _p],
    "sci_bayer4_to_mosaic": [_p, _p, _i, _i, _i, _p],
    "sci_mosaic_to_bayer4": [_p, _p, _i, _i, _i, _p],
    "sci_psnr_accum": [_p, _p, _l, _i, _p, _p],
    "sci_ssim_accum": [_p, _p, _i, _i, _i, _d, _p, _p],
    "sci_conv_tc_available": [],
    "sci_conv3x3_fwd": [_p, _i, _p],
    "sci_conv3x3_dgrad": [_p, _i, _p],
    "sci_conv3x3_wgrad": [_p, _i, _p],
    "sci_conv_pack_weights": [_p, _p, _i, _i, _i, _i, _i, _i, _p, _i, _i, _i, _p],
    "sci_conv_pack_weights_s2t": [_p, _p, _i, _i, _i, _i, _p, _i, _p],
    "sci_conv_pack_weights_half": [_p, _p, _i, _i, _i, _i, _i, _i, _i, _p],
    "sci_layer_ops_batch": [_p, _i, _i, _p],
    "sci_p2p_alloc": [_sz, _p],
    "sci_p2p_free": [_p],
    "sci_p2p_get_handle": [_p, _p],
    "sci_p2p_open_handle": [_p, _p],
    "sci_p2p_close_handle": [_p],
    "sci_halo_send": [_p, _i, _i, _i, _i, _p, _p, _p, _p, ctypes.c_uint, _p, _p],
    "sci_halo_send_tv": [_p, _p, _f, _i, _i, _i, _i, _p, _p, _p, _p, ctypes.c_uint, _p, _p],
    "sci_halo_assemble": [_p, _i, _i, _i, _i, _i, _p, _p, _p, _p, ctypes.c_uint, _p, _p, _p],
    "sci_fastdvd_pack_input_half": [_p, _f, _p, _i, _i, _i, _i, _p],
    "sci_fastdvd_pack_input_half_planes": [_p, _f, _p, _i, _i, _i, _i, _i, _p],
    "sci_conv_unpack_wgrad": [_p, _p, _i, _i, _i, _i, _i, _i, _i, _p],
    "sci_bn_fold": [_p, _p, _p, _p, _f, _p, _p, _i, _i, _p],
    "sci_act_bwd": [_p, _p, _p, _l, _i, _i, _p, _p, _p],
    "sci_act_bwd_ordered": [_p, _p, _p, _l, _i, _i, _p, _p, _p, _sz, _p],
    "sci_bn_param_grad": [_p, _p, _p, _p, _p, _p, _i, _p],
    "sci_nhwc_pixel_unshuffle": [_p, _p, _i, _i, _i, _i, _p],
    "sci_nhwc_dilate2": [_p, _p, _i, _i, _i, _i, _p],
    "sci_ffdnet_pack_input": [_p, _f, _p, _i, _i, _i, _i, _i, _i, _p],
    "sci_ffdnet_unpack_output": [_p, _p, _i, _i, _i, _i, _i, _p],
    "sci_ffdnet_unpack_output_grad": [_p, _p, _i, _i, _i, _i, _i, _p],
    "sci_ffdnet_pack_input_split_half": [_p, _f, _p, _i, _i, _i, _i, _p],
    "sci_ffdnet_unpack_output_split_half": [_p, _p, _i, _i, _i, _i, _p],
    "sci_dual_update_gray": [_p, _p, _p, _p, _p, _p, _i, _l, _p, _p, _p],
    "sci_fastdvd_pack_input": [_p, _f, _p, _i, _i, _i, _i, _i, _p],
    "sci_fastdvd_output": [_p, _p, _p, _i, _i, _i, _i, _p],
    "sci_fastdvd_output_grad": [_p, _p, _i, _i, _i, _i, _p],
    "sci_fastdvd_pack_input_grad": [_p, _p, _i, _i, _i, _i, _i, _p],
    "sci_fastdvd_pack_input_planes": [_p, _f, _p, _i, _i, _i, _i, _i, _i, _p],
    "sci_fastdvd_output_planes": [_p, _p, _p, _i, _i, _i, _i, _i, _p],
    "sci_fastdvd_output_grad_planes": [_p, _p, _i, _i, _i, _i, _i, _p],
    "sci_fastdvd_pack_input_grad_planes": [_p, _p, _i, _i, _i, _i, _i, _i, _p],
    "sci_fastdvd_noisy_input": [_p, _p, _p, _l, _p],
    "sci_rgb_sum": [_p, _p, _i, _i, _i, _p],
    "sci_ddnet_pack_input1": [_p, _p, _p, _i, _i, _i, _i, _i, _p],
    "sci_ddnet_pack_input4": [_p, _p, _p, _i, _i, _i, _i, _i, _p],
    "sci_ddnet_stage2_input": [_p, _p, _p, _i, _p, _p, _i, _i, _i, _i, _i, _p],
    "sci_ddnet_upsample4": [_p, _p, _p, _i, _p, _i, _i, _i, _i, _i, _p],
    "sci_ddnet_output": [_p, _p, _p, _i, _p, _p, _i, _i, _i, _p],
    "sci_ddnet_pack_input1_frames": [_p, _p, _p, _i, _i, _i, _i, _i, _i, _i, _p],
    "sci_ddnet_pack_input4_frames": [_p, _p, _p, _i, _i, _i, _i, _i, _i, _i, _p],
    "sci_ddnet_stage2_input_frames": [_p, _p, _p, _i, _p, _p, _i, _i, _i, _i, _i, _i, _i, _p],
    "sci_ddnet_upsample4_strip": [_p, _p, _p, _i, _p, _i, _i, _i, _i, _i, _i, _i, _i, _i, _p],
    "sci_ddnet_loss_fwd_bwd": [_p, _p, _p, _p, _i, _i, _i, _p],
    "sci_ddnet_output_bwd": [_p, _p, _p, _p, _i, _p, _p, _p, _p, _p, _i, _i, _i, _p],
    "sci_ddnet_stage2_input_bwd": [_p, _p, _p, _p, _p, _i, _i, _i, _p],
    "sci_ddnet_pack_input1_bwd": [_p, _p, _p, _i, _i, _i, _p],
    "sci_ddnet_pack_input4_bwd": [_p, _p, _p, _i, _i, _i, _i, _p],
    "sci_ddnet_upsample4_bwd": [_p, _p, _i, _i, _i, _p],
    "sci_host_legacy_normal": [_p, _p, _p, _p, _d, _d, _p, _l, _i],
    "sci_meas_loss_fwd_bwd": [_p, _p, _p, _p, _p, _i, _i, _i, _i, _l, _p],
    "sci_axpy": [_p, _f, _p, _p, _l, _p],
    "sci_adam_step": [_p, _p, _p, _p, _l, _d, _d, _d, _d, _i, _p],
}
_SPECIAL_RESTYPE = {"sci_last_error": ctypes.c_char_p, "sci_tv_workspace_bytes": _sz, "sci_tv_strip_workspace_bytes": _sz,
                    "sci_conv3x3_fwd_workspace_bytes": _sz, "sci_conv3x3_wgrad_workspace_bytes": _sz,
                    "sci_act_bwd_workspace_bytes": _sz}

for _name, _args in PROTOTYPES.items():
    _fn = getattr(lib, _name)
    _fn.argtypes = _args
    _fn.restype = _i
lib.sci_last_error.argtypes = []
lib.sci_last_error.restype = ctypes.c_char_p
lib.sci_tv_workspace_bytes.argtypes = [_i, _i, _i]
lib.sci_tv_workspace_bytes.restype = _sz
lib.sci_tv_strip_workspace_bytes.argtypes = [_i, _i, _i]
lib.sci_tv_strip_workspace_bytes.restype = _sz
lib.sci_conv3x3_fwd_workspace_bytes.argtypes = [_p, _i]
lib.sci_conv3x3_fwd_workspace_bytes.restype = _sz
lib.sci_conv3x3_wgrad_workspace_bytes.argtypes = [_p, _i]
lib.sci_conv3x3_wgrad_workspace_bytes.restype = _sz
lib.sci_act_bwd_workspace_bytes.argtypes = [_l, _i]
lib.sci_act_bwd_workspace_bytes.restype = _sz


class SciError(RuntimeError):
    pass


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    if t is None:
        return None
    return ctypes.c_void_p(t.data_ptr())


def stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def check(rc, what):
    if rc != 0:
        msg = lib.sci_last_error()
        raise SciError("%s failed (code %d): %s" % (what, rc, msg.decode() if msg else ""))


# kernel launches issued through the C ABI since import (bench.py reports the count inside its timed region)
KERNELS_PER_CALL = {"sci_tv_chambolle2d": 3, "sci_tv_strip_main": 2, "sci_tv_strip_finish": 2, "sci_version": 0,
                    "sci_conv_tc_available": 0, "sci_host_legacy_normal": 0, "sci_act_bwd_ordered": 2}
launch_count = 0


def call(name, *args):
    global launch_count
    check(getattr(lib, name)(*args), name)
    launch_count += KERNELS_PER_CALL.get(name, 1)


def require_cuda_f32(*tensors):
    for t in tensors:
        if t is None:
            continue
        if not (t.is_cuda and t.dtype == torch.float32 and t.is_contiguous()):
            raise SciError("expected contiguous float32 CUDA tensors, got %s %s contiguous=%s"
                           % (t.device, t.dtype, t.is_contiguous()))
