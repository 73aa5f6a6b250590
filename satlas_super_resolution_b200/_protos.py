"""ctypes prototypes for the entry points of include/ssr_b200.h beyond the conv core."""
import ctypes as C

i32, f32, vp = C.c_int32, C.c_float, C.c_void_p


class PackDesc(C.Structure):
    """Mirror of struct ssr_pack_desc."""
    _fields_ = [("w", vp), ("dst", vp), ("inv_scale", vp),
                ("cout", i32), ("cin", i32), ("r", i32), ("mode", i32), ("k_pad", i32), ("n_pad", i32)]


class WgradArgs(C.Structure):
    """Mirror of struct ssr_wgrad_tc_args."""
    _fields_ = [("x", vp), ("n_img", i32), ("h", i32), ("w", i32), ("x_pix_stride", i32), ("cx", i32),
                ("dy", vp), ("dy_pix_stride", i32), ("cy", i32), ("r", i32),
                ("out", vp), ("out_cx_rows", i32), ("out_stride", i32), ("scale", f32), ("splits", i32)]


class UnpackDesc(C.Structure):
    """Mirror of struct ssr_unpack_desc."""
    _fields_ = [("acc", vp), ("grad", vp), ("cx_rows", i32), ("acc_stride", i32), ("cout", i32), ("cin", i32), ("r", i32),
                ("accumulate", i32), ("scale", f32), ("pad_", i32)]


class SnDesc(C.Structure):
    """Mirror of struct ssr_sn_desc."""
    _fields_ = [("w", vp), ("u", vp), ("v", vp), ("sigma", vp), ("scratch", vp), ("geff", vp), ("grad", vp),
                ("rows", i32), ("cols", i32)]


i64 = C.c_int64
PROTOS = {
    "ssr_profile_start": (C.c_int, []),
    "ssr_profile_stop": (C.c_int, [vp, vp, i32]),
    "ssr_im2col": (C.c_int, [vp, i32, vp, i32, i32, i32, i32, i32, i32, i32, vp]),
    "ssr_col2im": (C.c_int, [vp, vp, i32, i32, i32, i32, i32, i32, i32, i32, vp, i32, vp, i32, vp]),
    "ssr_axpby": (C.c_int, [vp, i32, f32, vp, i32, f32, vp, i32, i32, vp, i32, i64, i32, vp]),
    "ssr_maxpool_relu": (C.c_int, [vp, vp, i32, i32, i32, i32, vp]),
    "ssr_feat_grad": (C.c_int, [vp, vp, vp, i32, i32, i32, i32, f32, vp]),
    "ssr_feat_l1": (C.c_int, [vp, i64, f32, vp, vp]),
    "ssr_l1_loss": (C.c_int, [vp, vp, i64, f32, vp, vp, i32, vp]),
    "ssr_pack_tile_count": (C.c_int32, [i32, i32]),
    "ssr_pack_conv_weights_tiled": (C.c_int, [vp, vp, i32, vp]),
    "ssr_split_finish": (C.c_int, [vp, vp, vp, i32, i64, i32, vp, i32, f32, vp, i32, f32, vp, i32, f32, vp, i32, vp, i32, vp, vp, i32, i32, vp]),
    "ssr_sum_pool2x2_f32": (C.c_int, [vp, vp, i32, i32, i32, i32, vp]),
    "ssr_ssim_loss": (C.c_int, [vp, vp, i32, i32, i32, f32, vp, vp, i32, vp, vp]),
    "ssr_bce_logits": (C.c_int, [vp, i64, f32, f32, vp, vp, vp, vp]),
    "ssr_disc_input": (C.c_int, [vp, i32, vp, i32, i32, i32, vp, i32, i32, i32, i32, vp]),
    "ssr_disc_input_ex": (C.c_int, [vp, i32, vp, i32, i32, i32, vp, i32, vp, i32, i32, i32, i32, vp]),
    "ssr_ema_update": (C.c_int, [vp, vp, i64, f32, vp]),
    "ssr_ingest_nchw_unshuffle": (C.c_int, [vp, vp, i32, i32, i32, i32, i32, i32, i32, f32, vp]),
    "ssr_f32_nchw_to_u8_hwc": (C.c_int, [vp, vp, i32, i32, i32, i32, i32, vp]),
    "ssr_u8_shift_diff_sums": (C.c_int, [vp, vp, i32, i32, i32, i32, i32, i32, vp, vp]),
    "ssr_u8_ssim_sums": (C.c_int, [vp, vp, i32, i32, i32, i32, i32, vp, vp, vp]),
    "ssr_ingest_u8_nhwc": (C.c_int, [vp, i32, i32, i32, i32, vp, i32, i32, i32, vp, vp, vp]),
    "ssr_lpips_cta_count": (C.c_int32, [i32, i32]),
    "ssr_lpips_layer_sums": (C.c_int, [vp, i32, i32, i32, i32, vp, vp, vp]),
    "ssr_lpips_finish": (C.c_int, [vp, i32, i32, C.POINTER(i32), C.POINTER(i32), vp, vp]),
    "ssr_spectral_norm": (C.c_int, [vp, i32, i32, f32, vp]),
    "ssr_spectral_norm_bwd": (C.c_int, [vp, i32, vp]),
    "ssr_usm_sharp": (C.c_int, [vp, vp, vp, i32, i32, i32, vp, i32, f32, f32, vp]),
    "ssr_u8_to_f32": (C.c_int, [vp, vp, i64, f32, vp]),
    "ssr_adam_tick": (C.c_int, [vp, vp]),
    "ssr_adam_ema": (C.c_int, [vp, vp, vp, vp, vp, i64, f32, f32, f32, f32, f32, i32, f32, f32, vp, vp]),
    "ssr_debug_chain_timeline": (C.c_int, [vp, i32]),
    "ssr_debug_resident_launches": (C.c_int64, []),
    "ssr_debug_conv_path_count": (C.c_int64, [i32]),
    "ssr_wgrad_tc": (C.c_int, [C.POINTER(WgradArgs), vp]),
    "ssr_wgrad_tc_batched": (C.c_int, [C.POINTER(WgradArgs), i32, vp]),
    "ssr_wgrad_unpack": (C.c_int, [vp, i32, i32, vp, i32, i32, i32, f32, i32, vp]),
    "ssr_bias_grad": (C.c_int, [vp, i32, C.c_int64, i32, vp, f32, vp]),
    "ssr_bias_grad_groups": (C.c_int, [vp, i32, C.c_int64, i32, i32, vp, f32, vp]),
    "ssr_ingest_nchw": (C.c_int, [vp, i32, vp, i32, i32, i32, i32, i32, i32, f32, vp, vp, vp]),
    "ssr_f32_nchw_to_u8_canvas": (C.c_int, [vp, vp, i32, i32, i32, i32, i32, i32, i32, vp]),
    "ssr_egress_nchw": (C.c_int, [vp, i32, vp, i32, i32, i32, i32, f32, i32, vp, vp]),
    "ssr_upsample_nearest": (C.c_int, [vp, i32, vp, i32, i32, i32, i32, i32, i32, vp]),
    "ssr_upsample_nearest_bwd": (C.c_int, [vp, i32, vp, i32, i32, i32, i32, i32, i32, vp, i32, vp]),
    "ssr_upsample_bilinear2x": (C.c_int, [vp, i32, vp, i32, vp, i32, i32, i32, i32, i32, vp]),
    "ssr_upsample_bilinear2x_bwd": (C.c_int, [vp, i32, vp, i32, i32, i32, i32, i32, vp]),
    "ssr_pack_conv_weights_batched": (C.c_int, [vp, i32, i32, vp]),
    "ssr_wgrad_unpack_batched": (C.c_int, [vp, i32, vp]),
}


def bind(lib):
    for name, (restype, argtypes) in PROTOS.items():
        fn = getattr(lib, name, None)
        if fn is None:
            raise AttributeError(f"libssr_b200.so does not export {name} (stale build?)")
        fn.restype = restype
        fn.argtypes = argtypes
