"""ctypes binding of libmega_b200.so (the C ABI declared in include/mega_b200.h).

The library is the product: if it is missing or does not load, importing this module raises --
there is no CPU or PyTorch fallback anywhere in the package.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
_PKG_ROOT = os.path.dirname(_HERE)
LIB_PATH = os.environ.get("MEGA_B200_LIB", os.path.join(_PKG_ROOT, "lib", "libmega_b200.so"))

if not os.path.exists(LIB_PATH):
    raise ImportError(
        "libmega_b200.so not found at %s -- run `python mega.pytorch_b200/build.py` "
        "(or __graft_entry__.build()) first; there is no fallback path" % LIB_PATH)

lib = ctypes.CDLL(LIB_PATH)

c_f32p = ctypes.c_void_p
c_ll = ctypes.c_longlong
c_int = ctypes.c_int


class ConvGemmDesc(ctypes.Structure):
    """mirror of `mega_conv_gemm_desc` (include/mega_b200.h)"""
    _fields_ = [
        ("a", c_f32p),
        ("a_n", c_int), ("a_h", c_int), ("a_w", c_int), ("a_c", c_int),
        ("a_stride_w", c_ll), ("a_stride_h", c_ll), ("a_stride_n", c_ll),
        ("b", c_f32p),
        ("b_n", c_int), ("b_k", c_int),
        ("b_stride_n", c_ll), ("b_stride_tap", c_ll),
        ("taps_r", c_int), ("taps_s", c_int), ("dil", c_int), ("pad", c_int),
        ("k_per_tap", c_int),
        ("out", c_f32p),
        ("out_ld", c_ll),
        ("n_img", c_int), ("out_h", c_int), ("out_w", c_int), ("cout", c_int),
        ("scale", c_f32p), ("bias", c_f32p), ("residual", c_f32p),
        ("res_ld", c_ll),
        ("relu", c_int),
        ("tile_h", c_int), ("tile_w", c_int), ("block_n", c_int),
        ("batch", c_int),
        ("a_c_off", c_int), ("a_n_off", c_int), ("b_k_off", c_int), ("b_n_off", c_int),
        ("out_c_off", c_int), ("out_n_off", c_int), ("res_c_off", c_int), ("res_n_off", c_int),
        ("bias_z_off", c_int),
        ("precision", c_int),
        ("max_ctas", c_int),
        ("stream_k", c_int),
        ("workspace", ctypes.c_void_p),
        ("workspace_bytes", c_ll),
        ("out_f16", c_int),
        ("pdl", c_int),
        ("stride_h", c_int), ("stride_w", c_int), ("pad_w_set", c_int), ("pad_w", c_int),
        ("out_stride_h", c_ll), ("out_stride_n", c_ll), ("res_stride_h", c_ll), ("res_stride_n", c_ll),
        ("b_lo_tap_off", c_int), ("res_split", c_int), ("acc_scale", ctypes.c_float), ("reserved_v6", c_int),
    ]


lib.mega_last_error.restype = ctypes.c_char_p
lib.mega_abi_version.restype = c_int
lib.mega_device_ok.restype = c_int
lib.mega_conv_gemm.argtypes = [ctypes.POINTER(ConvGemmDesc), ctypes.c_void_p]
lib.mega_conv_gemm.restype = c_int
lib.mega_conv_gemm_tf32.argtypes = [ctypes.POINTER(ConvGemmDesc), ctypes.c_void_p]
lib.mega_conv_gemm_tf32.restype = c_int
lib.mega_conv_gemm_workspace_bytes.restype = c_ll
lib.mega_conv_chain_plan_bytes.argtypes = [c_int]
lib.mega_conv_chain_plan_bytes.restype = c_ll
lib.mega_conv_chain_encode.argtypes = [ctypes.POINTER(ConvGemmDesc), c_int, ctypes.c_void_p, c_ll, ctypes.POINTER(c_int)]
lib.mega_conv_chain_encode.restype = c_int
lib.mega_conv_chain_launch.argtypes = [ctypes.c_void_p, c_int, c_int, ctypes.c_void_p, ctypes.c_void_p, c_int]
lib.mega_conv_chain_launch.restype = c_int
lib.mega_conv_chain_encode2.argtypes = [ctypes.POINTER(ConvGemmDesc), c_int, ctypes.c_void_p, c_ll, ctypes.POINTER(c_int), c_int]
lib.mega_conv_chain_encode2.restype = c_int
lib.mega_conv_chain_launch2.argtypes = [ctypes.c_void_p, c_int, c_int, ctypes.c_void_p, ctypes.c_void_p, c_int, c_int]
lib.mega_conv_chain_launch2.restype = c_int
lib.mega_conv_chain_set_trace.argtypes = [ctypes.c_void_p, c_int]
lib.mega_conv_chain_set_trace.restype = c_int
lib.mega_conv_chain_set_trace2.argtypes = [ctypes.c_void_p, c_int, c_int]
lib.mega_conv_chain_set_trace2.restype = c_int
lib.mega_nms_host.argtypes = [ctypes.c_void_p, ctypes.c_void_p, c_int, ctypes.c_float, c_int, ctypes.c_void_p, ctypes.c_void_p]
lib.mega_nms_host.restype = c_int
lib.mega_roi_align_forward_nchw_host.argtypes = [ctypes.c_void_p, c_int, c_int, c_int, c_int, ctypes.c_void_p, c_int,
                                                 ctypes.c_float, c_int, c_int, c_int, c_int, ctypes.c_void_p]
lib.mega_roi_align_forward_nchw_host.restype = c_int
lib.mega_set_split16_a_tmem.argtypes = [c_int]
lib.mega_set_split16_a_tmem.restype = c_int
lib.mega_set_split3_seg_len.argtypes = [c_int]
lib.mega_set_split3_seg_len.restype = c_int
lib.mega_set_tf32_rounding.argtypes = [c_int]
lib.mega_set_tf32_rounding.restype = c_int


class MegaError(RuntimeError):
    pass


def check(status, what=""):
    if status != 0:
        msg = lib.mega_last_error().decode("utf-8", "replace")
        raise MegaError("%s failed (status %d): %s" % (what or "libmega_b200 call", status, msg))


def stream_ptr():
    """cudaStream_t of torch's current stream, as an integer for ctypes."""
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    if t is None:
        return None
    return ctypes.c_void_p(t.data_ptr())


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise MegaError("libmega_b200 ops take CUDA tensors only (got a %s tensor); "
                            "the B200 path has no CPU fallback" % t.device)


# ---- argtypes of the remaining entry points (include/mega_b200.h)
_vp, _i, _f, _ll = ctypes.c_void_p, ctypes.c_int, ctypes.c_float, ctypes.c_longlong
lib.mega_nms_workspace_bytes.argtypes = [_i]
lib.mega_nms_workspace_bytes.restype = _ll
lib.mega_nms.argtypes = [_vp, _vp, _i, _f, _vp, _ll, _vp, _vp, _vp]
lib.mega_nms.restype = _i
lib.mega_rpn_select_workspace_bytes.argtypes = [_i, _i, _i, _i, _i]
lib.mega_rpn_select_workspace_bytes.restype = _ll
lib.mega_rpn_select.argtypes = [_vp, _ll, _i, _i, _i, _i, _i, _i, _vp, _f, _f, _i, _i, _f, _f, _vp, _ll, _vp, _vp,
                                _vp, _vp, _vp]
lib.mega_rpn_select.restype = _i
lib.mega_roi_align_forward_nchw.argtypes = [_vp, _i, _i, _i, _i, _vp, _i, _f, _i, _i, _i, _vp, _vp]
lib.mega_roi_align_forward_nchw.restype = _i
lib.mega_roi_align_forward_nhwc.argtypes = [_vp, _i, _i, _i, _ll, _vp, _i, _i, _vp, _i, _f, _i, _i, _i, _vp, _ll, _vp]
lib.mega_roi_align_forward_nhwc.restype = _i
lib.mega_roi_align_forward_nhwc_f16.argtypes = [_vp, _i, _i, _i, _ll, _vp, _i, _i, _vp, _i, _f, _i, _i, _i, _vp, _ll, _vp]
lib.mega_roi_align_forward_nhwc_split16.argtypes = [_vp, _i, _i, _i, _ll, _vp, _i, _i, _vp, _i, _f, _i, _i, _i, _vp, _ll, _vp]
lib.mega_roi_align_forward_nhwc_split16.restype = _i
lib.mega_roi_align_forward_nhwc_f16.restype = _i
lib.mega_stem_im2col_f16.argtypes = [_vp, _i, _i, _i, _i, _vp, _vp]
lib.mega_stem_im2col_f16.restype = _i
lib.mega_maxpool3x3s2_nhwc_f16.argtypes = [_vp, _i, _i, _i, _i, _vp, _vp]
lib.mega_maxpool3x3s2_nhwc_f16.restype = _i
lib.mega_relation_softmax_f16.argtypes = [_vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _i, _f, _vp]
lib.mega_relation_softmax_split16.argtypes = [_vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _i, _f, _vp]
lib.mega_relation_softmax_split16.restype = _i
lib.mega_relation_softmax_f16.restype = _i
lib.mega_relation_softmax_pe.argtypes = [_vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _i, _f, _vp]
lib.mega_relation_softmax_pe_split16.argtypes = [_vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _i, _f, _vp]
lib.mega_relation_softmax_pe_split16.restype = _i
lib.mega_relation_softmax_pe.restype = _i
lib.mega_fgfa_pool_image.argtypes = [_vp, _i, _i, _vp, _i, _vp]
lib.mega_fgfa_pool_image.restype = _i
lib.mega_fgfa_build_pairs.argtypes = [_vp, _ll, _vp, _i, _i, _i, _i, _vp, _i, _vp]
lib.mega_fgfa_build_pairs.restype = _i
lib.mega_avgpool2_nhwc.argtypes = [_vp, _i, _i, _i, _i, _ll, _vp, _ll, _i, _vp]
lib.mega_avgpool2_nhwc.restype = _i
lib.mega_fgfa_aggregate.argtypes = [_vp, _ll, _i, _i, _i, _vp, _i, _i, _vp, _i, _i, _i, _vp, _ll, _vp, _i, _vp]
lib.mega_fgfa_aggregate.restype = _i
lib.mega_stem_prep.argtypes = [_vp, _i, _i, _i, _i, _vp, _i, _vp]
lib.mega_stem_prep.restype = _i
lib.mega_stem_im2col.argtypes = [_vp, _i, _i, _i, _i, _vp, _vp]
lib.mega_stem_im2col.restype = _i
lib.mega_maxpool3x3s2_nhwc.argtypes = [_vp, _i, _i, _i, _i, _vp, _vp]
lib.mega_maxpool3x3s2_nhwc.restype = _i
lib.mega_gather_rows.argtypes = [_vp, _ll, _vp, _i, _i, _vp, _ll, _vp]
lib.mega_gather_rows.restype = _i
lib.mega_copy_rows.argtypes = [_vp, _ll, _vp, _vp, _ll, _vp, _i, _i, _vp]
lib.mega_copy_rows.restype = _i
class CopyJob(ctypes.Structure):
    """mirror of `mega_copy_job`"""
    _fields_ = [("src", ctypes.c_void_p), ("src_ld", ctypes.c_longlong), ("src_idx", ctypes.c_void_p),
                ("dst", ctypes.c_void_p), ("dst_ld", ctypes.c_longlong), ("dst_idx", ctypes.c_void_p),
                ("n_rows", ctypes.c_int), ("row_len", ctypes.c_int)]


lib.mega_copy_rows_batch.argtypes = [ctypes.POINTER(CopyJob), _i, _vp]
lib.mega_copy_rows_batch.restype = _i
lib.mega_split16_pack.argtypes = [_vp, _vp, _ll, _vp]
lib.mega_split16_pack.restype = _i
lib.mega_split16_unpack.argtypes = [_vp, _vp, _ll, _vp]
lib.mega_split16_unpack.restype = _i
lib.mega_transpose_2d.argtypes = [_vp, _i, _i, _i, _vp, _vp]
lib.mega_transpose_2d.restype = _i
lib.mega_relation_softmax.argtypes = [_vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _i, _f, _vp]
lib.mega_relation_softmax.restype = _i
lib.mega_box_postprocess_workspace_bytes.argtypes = [_i, _i]
lib.mega_box_postprocess_workspace_bytes.restype = _ll
lib.mega_box_postprocess.argtypes = [_vp, _i, _vp, _i, _vp, _vp, _i, _i, _f, _f, _f, _f, _i, _f, _f, _f, _f, _vp, _ll,
                                     _vp, _vp, _vp, _i, _vp, _vp]
lib.mega_box_postprocess.restype = _i

lib.mega_sigmoid_focalloss_forward.argtypes = [_vp, _vp, _i, _i, _f, _f, _vp, _vp]
lib.mega_sigmoid_focalloss_forward.restype = _i
lib.mega_sigmoid_focalloss_backward.argtypes = [_vp, _vp, _vp, _i, _i, _f, _f, _vp, _vp]
lib.mega_sigmoid_focalloss_backward.restype = _i
lib.mega_deform_im2col.argtypes = [_vp, _vp, _vp] + [_i] * 14 + [_vp, _vp]
lib.mega_deform_im2col.restype = _i
lib.mega_deform_psroi_pooling_forward.argtypes = [_vp, _vp, _vp, _i, _i, _i, _i, _i, _f, _i, _i, _i, _i, _i, _f, _i, _vp,
                                                  _vp, _vp]
lib.mega_deform_psroi_pooling_forward.restype = _i

# ---- ABI v4: training-side ops (csrc/train_ops.cu)
lib.mega_roi_align_backward_nchw.argtypes = [_vp, _vp, _i, _f, _i, _i, _i, _i, _i, _i, _i, _vp, _vp]
lib.mega_roi_align_backward_nchw.restype = _i
lib.mega_roi_pool_forward.argtypes = [_vp, _vp, _i, _f, _i, _i, _i, _i, _i, _vp, _vp, _vp]
lib.mega_roi_pool_forward.restype = _i
lib.mega_roi_pool_backward.argtypes = [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _vp]
lib.mega_roi_pool_backward.restype = _i
lib.mega_deform_im2col_kq.argtypes = [_vp, _vp, _vp] + [_i] * 14 + [_vp, _vp]
lib.mega_deform_im2col_kq.restype = _i
lib.mega_deform_col2im_fused.argtypes = [_vp, _vp, _vp, _vp] + [_i] * 14 + [_vp, _vp, _vp, _vp]
lib.mega_deform_col2im_fused.restype = _i
lib.mega_channel_sum_nchw.argtypes = [_vp, _i, _i, _i, _vp, _vp]
lib.mega_channel_sum_nchw.restype = _i
lib.mega_deform_psroi_pooling_backward.argtypes = [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _f, _i, _i, _i, _i, _i,
                                                   _f, _i, _vp, _vp, _vp]
lib.mega_deform_psroi_pooling_backward.restype = _i
lib.mega_image_transform_u8.argtypes = [_vp, _i, _i, _ll, _ll, _ll, _vp, _vp, _i, _vp, _vp, _i, _i, _i, _vp, _vp, _i, _vp, _vp]
lib.mega_image_transform_u8.restype = _i
lib.mega_dff_warp_scale.argtypes = [_vp, _i, _i, _vp, _i, _vp, _ll, _i, _i, _vp, _ll, _i, _vp]
lib.mega_dff_warp_scale.restype = _i
lib.mega_vid_match_host.argtypes = [_vp, _i, _vp, _vp, _i, _f, ctypes.c_double, _vp, _vp]
lib.mega_vid_match_host.restype = _i
lib.mega_vid_eval_workspace_bytes.argtypes = [_ll, _ll, _i, _i]
lib.mega_vid_eval_workspace_bytes.restype = _ll
lib.mega_vid_eval_match.argtypes = [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _ll, _ll, _i, _i, _vp, _vp, _f, _vp, _ll,
                                    _vp, _vp, _vp, _vp, _vp, _vp]
lib.mega_vid_eval_match.restype = _i
lib.mega_vid_eval_rank.argtypes = [_ll, _ll, _i, _i, _vp, _ll, _vp, _vp]
lib.mega_vid_eval_rank.restype = _i
lib.mega_vid_eval_scan_ap.argtypes = [_vp, _vp, _vp, _vp, _vp, _ll, _ll, _i, _i, _vp, _ll, _vp, _vp, _vp, _vp]
lib.mega_vid_eval_scan_ap.restype = _i

EXPORTS = [
    "mega_last_error", "mega_abi_version", "mega_device_ok", "mega_conv_gemm", "mega_conv_gemm_tf32", "mega_conv_gemm_workspace_bytes", "mega_set_tf32_rounding",
    "mega_conv_chain_plan_bytes", "mega_conv_chain_encode", "mega_conv_chain_launch", "mega_conv_chain_set_trace",
    "mega_conv_chain_encode2", "mega_conv_chain_launch2", "mega_set_split3_seg_len", "mega_set_split16_a_tmem", "mega_conv_chain_set_trace2", "mega_nms_host", "mega_roi_align_forward_nchw_host",
    "mega_nms_workspace_bytes", "mega_nms", "mega_rpn_select_workspace_bytes", "mega_rpn_select",
    "mega_roi_align_forward_nchw", "mega_roi_align_forward_nhwc", "mega_stem_im2col", "mega_maxpool3x3s2_nhwc",
    "mega_gather_rows", "mega_copy_rows", "mega_copy_rows_batch", "mega_transpose_2d", "mega_relation_softmax", "mega_box_postprocess_workspace_bytes",
    "mega_box_postprocess", "mega_sigmoid_focalloss_forward", "mega_sigmoid_focalloss_backward",
    "mega_deform_im2col", "mega_deform_psroi_pooling_forward",
    "mega_roi_align_forward_nhwc_f16", "mega_stem_im2col_f16", "mega_maxpool3x3s2_nhwc_f16", "mega_relation_softmax_f16", "mega_relation_softmax_pe",
    "mega_stem_prep", "mega_fgfa_pool_image", "mega_fgfa_build_pairs", "mega_avgpool2_nhwc", "mega_fgfa_aggregate",
    "mega_roi_align_backward_nchw", "mega_roi_pool_forward", "mega_roi_pool_backward", "mega_deform_im2col_kq",
    "mega_deform_col2im_fused", "mega_channel_sum_nchw", "mega_deform_psroi_pooling_backward",
    "mega_image_transform_u8", "mega_dff_warp_scale", "mega_vid_match_host", "mega_split16_pack", "mega_split16_unpack", "mega_relation_softmax_split16", "mega_relation_softmax_pe_split16", "mega_roi_align_forward_nhwc_split16",
    "mega_vid_eval_workspace_bytes", "mega_vid_eval_match", "mega_vid_eval_rank", "mega_vid_eval_scan_ap",
]
