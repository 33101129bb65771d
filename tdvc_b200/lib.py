"""ctypes binding of the C-ABI in include/tdvc_b200.h (tdvc_b200/libtdvc_b200.so).

There is no CPU fallback: if the library is missing this module raises at first use, and every wrapper
raises RuntimeError with the library's own message when a call returns a non-zero code (the reference
raises RuntimeError through AT_ASSERTM, reference main/utils/dcnv2/src/cuda/dcn_v2_cuda.cu:38-62).
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("TDVC_B200_LIB") or os.path.join(HERE, "libtdvc_b200.so")   # override: developer A/B builds only

ACT_NONE, ACT_RELU, ACT_LRELU, ACT_CLAMP01 = 0, 1, 2, 3
POST_NONE, POST_GDN, POST_IGDN = 0, 1, 2
IMPL_AUTO, IMPL_SIMT, IMPL_TC, IMPL_SMALL = 0, 1, 2, 3

c_fp = C.c_void_p  # device pointers travel as integers


class ConvParams(C.Structure):
    _fields_ = [("src", c_fp * 4), ("src_c", C.c_int32 * 4), ("src_ld", C.c_int32 * 4), ("n_src", C.c_int32),
                ("N", C.c_int32), ("H", C.c_int32), ("W", C.c_int32), ("Ho", C.c_int32), ("Wo", C.c_int32),
                ("weight", c_fp), ("bias", c_fp),
                ("cin", C.c_int32), ("cin_pad", C.c_int32), ("cout", C.c_int32), ("cout_pad", C.c_int32),
                ("kh", C.c_int32), ("kw", C.c_int32), ("stride", C.c_int32), ("pad", C.c_int32),
                ("in_square", C.c_int32), ("act", C.c_int32), ("slope", C.c_float), ("post", C.c_int32),
                ("mul", c_fp), ("mul_ld", C.c_int32), ("res1", c_fp), ("res1_ld", C.c_int32),
                ("res2", c_fp), ("res2_ld", C.c_int32), ("out", c_fp), ("out_ld", C.c_int32),
                ("shuffle", C.c_int32), ("impl", C.c_int32), ("weight_f16", c_fp), ("chan_sum", c_fp),
                ("w_shift", C.c_int32), ("order", C.c_int32), ("out_planar", C.c_int32),
                ("out_absmax", c_fp), ("in_absmax", c_fp), ("products", C.c_int32)]


class DcnParams(C.Structure):
    _fields_ = [("input", c_fp), ("in_ld", C.c_int32), ("offset", c_fp), ("off_ld", C.c_int32),
                ("mask", c_fp), ("mask_ld", C.c_int32), ("mask_is_logit", C.c_int32),
                ("weight_packed", c_fp), ("bias", c_fp), ("out", c_fp), ("out_ld", C.c_int32),
                ("N", C.c_int32), ("H", C.c_int32), ("W", C.c_int32), ("C", C.c_int32), ("O", C.c_int32),
                ("O_pad", C.c_int32), ("dg", C.c_int32), ("round_fp16", C.c_int32), ("act", C.c_int32),
                ("slope", C.c_float), ("impl", C.c_int32), ("weight_f16", c_fp), ("input_gp", c_fp),
                ("params_planar", C.c_int32)]


class ArChain(C.Structure):
    _fields_ = [("params", c_fp), ("params_ld", C.c_int32),
                ("w_ctx", c_fp), ("b_ctx", c_fp), ("w1", c_fp), ("b1", c_fp), ("c1", C.c_int32), ("c1_pad", C.c_int32),
                ("w2", c_fp), ("b2", c_fp), ("c2", C.c_int32), ("c2_pad", C.c_int32), ("w3", c_fp), ("b3", c_fp),
                ("scale_table", c_fp), ("n_scales", C.c_int32), ("y_hat", c_fp), ("symbols", c_fp), ("indexes", c_fp),
                ("N", C.c_int32), ("H", C.c_int32), ("W", C.c_int32), ("C", C.c_int32)]


class ArParams(C.Structure):
    _fields_ = [("chain", ArChain), ("y", c_fp), ("y_ld", C.c_int32), ("cluster", C.c_int32), ("cluster_used_host", c_fp)]


class ArDecodeParams(C.Structure):
    _fields_ = [("chain", ArChain), ("words", c_fp), ("word_offsets", c_fp),
                ("cdfs", c_fp), ("cdf_stride", C.c_int32), ("cdf_lengths", c_fp), ("cdf_offsets", c_fp),
                ("n_tables", C.c_int32), ("cdf_total", C.c_int32), ("status", c_fp), ("cluster", C.c_int32)]


i32, i64, f32, vp, sz = C.c_int32, C.c_int64, C.c_float, C.c_void_p, C.c_size_t

# name -> argtypes, in header order (tests check that every symbol declared in include/tdvc_b200.h is here)
SIGNATURES = {
    "tdvc_version": [],
    "tdvc_last_error": [],
    "tdvc_conv2d": [C.POINTER(ConvParams), vp],
    "tdvc_conv2d_f16_bytes": [C.POINTER(ConvParams)],
    "tdvc_conv2d_f16_is_split": [C.POINTER(ConvParams)],
    "tdvc_conv2d_products": [C.POINTER(ConvParams)],
    "tdvc_conv2d_chan_sum_rows": [C.POINTER(ConvParams)],
    "tdvc_conv2d_pack_f16": [C.POINTER(ConvParams), vp, vp],
    "tdvc_dcn_v2_workspace_bytes": [i32] * 6,
    "tdvc_dcn_v2_forward": [vp] * 6 + [i32] * 14 + [vp, sz, vp],
    "tdvc_dcn_v2_backward_workspace_bytes": [i32] * 8,
    "tdvc_dcn_v2_backward": [vp] * 10 + [i32] * 14 + [vp, sz, vp],
    "tdvc_dcn_nhwc": [C.POINTER(DcnParams), vp],
    "tdvc_dcn_f16_bytes": [i32],
    "tdvc_dcn_pack_f16": [vp, i32, i32, i32, vp, vp],
    "tdvc_nhwc_to_group_planar": [vp, i32, vp, i32, i32, i32, i32, vp],
    "tdvc_zero_bytes": [vp, sz, vp],
    "tdvc_slices_hash": [vp, i64, i64, i32, vp, vp],
    "tdvc_bpp_finish": [vp, vp, C.c_double, vp],
    "tdvc_nchw_to_nhwc": [vp, vp, i32, i32, i32, i32, i32, vp],
    "tdvc_nhwc_to_nchw": [vp, i32, vp, i32, i32, i32, i32, vp],
    "tdvc_avgpool2x2": [vp, vp, i32, i32, i32, i32, vp],
    "tdvc_spynet_prep": [vp, vp, vp, vp, i32, i32, i32, vp],
    "tdvc_spynet_prep_backward": [vp, vp, vp, vp, vp, i32, i32, i32, vp],
    "tdvc_upsample2x": [vp, vp, i32, i32, i32, i32, vp],
    "tdvc_add_flow_tiled": [vp, vp, vp, i32, i32, i32, i32, vp],
    "tdvc_axpby": [vp, vp, vp, i64, f32, f32, vp],
    "tdvc_bcast_add_lrelu": [vp, vp, vp, i32, i64, f32, vp],
    "tdvc_bcast_add_lrelu_multi": [C.POINTER(vp), vp, C.POINTER(vp), i32, i64, f32, vp],
    "tdvc_round_half_even": [vp, vp, i64, vp],
    "tdvc_se_partial_sums": [vp, i32, i32, i64, i32, vp, i32, vp],
    "tdvc_se_apply": [vp, i32, vp, i32, vp, vp, vp, vp, i32, i64, i32, i32, i32, f32, vp, i32, vp, i32, vp, i32, vp, i32, vp],
    "tdvc_eb_bits": [vp, vp, vp, vp, vp, vp, i64, i32, vp, vp],
    "tdvc_gc_bits": [vp, vp, i32, i64, i32, vp, vp],
    "tdvc_eb_bits_noise": [vp, vp, vp, vp, vp, vp, i64, i32, vp, vp],
    "tdvc_gc_bits_noise": [vp, vp, vp, i32, i64, i32, vp, vp],
    "tdvc_eb_aux_loss": [vp, vp, vp, vp, vp, i32, vp, vp],
    "tdvc_eb_aux_loss_grad": [vp, vp, vp, vp, vp, vp, i32, vp, vp],
    "tdvc_uniform_noise": [vp, i64, C.c_uint64, C.c_uint64, vp],
    "tdvc_uniform_noise_dev": [vp, i64, vp, C.c_uint64, vp],
    "tdvc_act_backward": [vp, vp, vp, i64, i32, f32, vp],
    "tdvc_zero_insert": [vp, i32, vp, i32, i32, i32, i32, i32, i32, i32, i32, vp],
    "tdvc_conv2d_wgrad_workspace_bytes": [i32] * 6,
    "tdvc_conv2d_wgrad": [vp, i32, vp, i32] + [i32] * 10 + [vp, vp, vp, sz, vp],
    "tdvc_conv2d_pack_weight": [vp, i32, i32, i32, i32, vp, i32, i32, vp, vp, vp],
    "tdvc_gdn_backward_pre": [vp, vp, vp, vp, vp, i64, i32, vp],
    "tdvc_gdn_backward_post": [vp, vp, vp, vp, i64, vp],
    "tdvc_chan_affine": [vp, vp, vp, vp, i32, i64, i32, vp],
    "tdvc_chan_dot_workspace_bytes": [i32, i64, i32],
    "tdvc_chan_dot": [vp, vp, vp, i32, i64, i32, f32, vp, sz, vp],
    "tdvc_pmf_to_quantized_cdf": [vp, i32, i32, vp],
    "tdvc_eb_symbols": [vp, i32, vp, i32, i32, i32, vp, vp, vp],
    "tdvc_ar_code_workspace_bytes": [i32, i32, i32],
    "tdvc_ar_code": [C.POINTER(ArParams), vp, sz, vp],
    "tdvc_ar_decode": [C.POINTER(ArDecodeParams), vp],
    "tdvc_rans_encode_with_indexes": [vp, vp, i64, vp, i32, vp, vp, i32, vp, i64],
    "tdvc_rans_decode_with_indexes": [vp, i64, vp, i64, vp, i32, vp, vp, i32, vp],
    "tdvc_gc_bits_backward": [vp, vp, vp, i32, vp, vp, vp, i64, i32, vp],
    "tdvc_eb_bits_backward": [vp, vp, vp, vp, vp, vp, vp, vp, vp, i64, i32, vp],
    "tdvc_avgpool_scale": [vp, i32, vp, i32, i32, i32, i32, i32, vp],
    "tdvc_ff_descriptors": [vp, vp, i32, i32, i32, i32, vp],
    "tdvc_ff_match": [vp, vp, vp, vp, i32, i32, i32, vp],
    "tdvc_ff_gather": [vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, vp],
    "tdvc_sq_err_sum": [vp, vp, i64, vp, vp],
    "tdvc_ssim_level": [vp, vp, i32, i32, i32, i32, C.POINTER(C.c_float), f32, f32, vp, vp],
    "tdvc_avgpool2_pad": [vp, vp, i32, i32, i32, vp],
}

_lib = None


def load():
    """Load the shared library once.  Raises (never falls back) when it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} not found: build it with `python -m tdvc_b200.build` "
                           "(tdvc_b200 has no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    for name, args in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.argtypes = args
        fn.restype = C.c_int
    lib.tdvc_last_error.restype = C.c_char_p
    lib.tdvc_dcn_v2_workspace_bytes.restype = C.c_size_t
    lib.tdvc_dcn_v2_backward_workspace_bytes.restype = C.c_size_t
    lib.tdvc_conv2d_f16_bytes.restype = C.c_size_t
    lib.tdvc_dcn_f16_bytes.restype = C.c_size_t
    lib.tdvc_ar_code_workspace_bytes.restype = C.c_size_t
    lib.tdvc_conv2d_wgrad_workspace_bytes.restype = C.c_size_t
    lib.tdvc_chan_dot_workspace_bytes.restype = C.c_size_t
    lib.tdvc_rans_encode_with_indexes.restype = C.c_int64
    _lib = lib
    return lib


def check(rc, what):
    if rc != 0:
        msg = load().tdvc_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"tdvc_b200: {what} failed ({rc}): {msg}")
