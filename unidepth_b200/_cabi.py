"""ctypes binding of libudb.so (include/udb.h).  Thin: structures mirror the C structs field for
field; every call raises RuntimeError with udb_last_error() on a non-zero return.  There is no
fallback: if the library is missing the import fails loudly."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("UDB_LIB", os.path.join(_HERE, "libudb.so"))   # UDB_LIB: alternative build (experiments)

A_MATRIX, A_CONV3X3 = 0, 1
ACT_NONE, ACT_GELU, ACT_LEAKY = 0, 1, 2
STORE_ROWS, STORE_CONVT, STORE_CONVTILE, STORE_HEAD = 0, 1, 2, 3

vp, i32, i64, f32 = C.c_void_p, C.c_int32, C.c_int64, C.c_float


class Gemm(C.Structure):
    _fields_ = [
        ("a", vp), ("w", vp), ("M", i32), ("N", i32), ("K", i32), ("lda", i32), ("ldw", i32),
        ("a_mode", i32),
        ("conv_B", i32), ("conv_H", i32), ("conv_W", i32), ("conv_C", i32), ("conv_inH", i32),
        ("conv_inW", i32), ("conv_off", i32), ("conv_TH", i32), ("conv_TW", i32),
        ("conv_cstride", i32), ("conv_coff", i32),
        ("bias", vp), ("gamma", vp), ("resid", vp), ("resid_f32", i32), ("out", vp), ("out_f32", i32),
        ("out2", vp), ("out2_leaky", i32), ("act", i32), ("store_mode", i32), ("ldc", i64),
        ("rows_per_group", i32), ("group_stride", i32), ("row_offset", i32),
        ("resid_mod", i32), ("resid_row_offset", i32), ("ldr", i64),
        ("ct_k", i32), ("ct_cout", i32), ("ct_h", i32), ("ct_w", i32), ("ct_pad", i32),
        ("head_w", vp), ("head_b", f32), ("head_add", f32),
        ("a_split_k", i32), ("out_split", i32),
        ("ln_stats_out", vp), ("ln_stats_in", vp), ("ln_c1", vp), ("ln_parts", i32), ("ln_part_cols", i32), ("ln_eps", f32),
    ]


class ConvHalo(C.Structure):
    _fields_ = [
        ("x", vp), ("w", vp), ("bias", vp),
        ("B", i32), ("H", i32), ("W", i32), ("C", i32), ("cstride", i32), ("coff", i32), ("cout", i32), ("act", i32),
        ("out", vp), ("ldc", i64), ("head_w", vp), ("head_b", f32), ("head_add", f32), ("head_out", vp),
    ]


class Attn(C.Structure):
    _fields_ = [
        ("q", vp), ("k", vp), ("v", vp), ("out", vp),
        ("B", i32), ("heads", i32), ("seq_q", i32), ("seq_k", i32), ("head_dim", i32),
        ("ldq", i32), ("ldk", i32), ("ldv", i32), ("ldo", i32),
        ("q_col0", i32), ("k_col0", i32), ("v_col0", i32), ("o_col0", i32), ("scale", f32),
        ("split", i32), ("lo_off_q", i32), ("lo_off_k", i32), ("lo_off_v", i32), ("lo_off_o", i32),
    ]


class LayerNorm(C.Structure):
    _fields_ = [
        ("inp", vp), ("in_f32", i32), ("out", vp), ("out_f32", i32), ("weight", vp), ("bias", vp),
        ("rows", i32), ("dim", i32), ("ld_in", i64), ("ld_out", i64),
        ("rows_per_group", i32), ("group_stride", i32), ("row_offset", i32), ("eps", f32), ("dim_valid", i32),
        ("out_split", i32),
    ]


class Preprocess(C.Structure):
    _fields_ = [
        ("rgb", vp), ("rgb_is_u8", i32), ("normalize", i32), ("B", i32), ("H", i32), ("W", i32),
        ("pad_l", i32), ("pad_r", i32), ("pad_t", i32), ("pad_b", i32), ("net_h", i32), ("net_w", i32),
        ("patches", vp), ("ldp", i32), ("split", i32),
    ]


class SmallLinear(C.Structure):
    _fields_ = [
        ("x", vp), ("w", vp), ("bias", vp), ("gamma", vp), ("resid", vp), ("y", vp),
        ("M", i32), ("N", i32), ("K", i32), ("act", i32), ("ldx", i32), ("ldy", i32), ("ldr", i32),
    ]


class RayEmbed(C.Structure):
    _fields_ = [
        ("intr4", vp), ("rays_in", vp), ("scales", vp),
        ("B", i32), ("net_h", i32), ("net_w", i32), ("gh", i32), ("gw", i32), ("bands", i32),
        ("out", vp), ("out_f32", i32),
    ]


class Postprocess(C.Structure):
    _fields_ = [
        ("radius", vp), ("confidence", vp), ("intr4", vp), ("rays_in", vp),
        ("B", i32), ("net_h", i32), ("net_w", i32), ("padded_h", i32), ("padded_w", i32),
        ("pad_l", i32), ("pad_t", i32), ("H", i32), ("W", i32),
        ("out_confidence", vp), ("out_radius", vp), ("out_depth", vp), ("out_points", vp), ("out_rays", vp),
    ]


class Config(C.Structure):
    _fields_ = [
        ("embed_dim", i32), ("depth", i32), ("enc_heads", i32), ("taps", i32 * 4), ("pos_grid", i32),
        ("hidden", i32), ("dec_heads", i32), ("expansion", i32), ("out_dim", i32), ("n_stages", i32),
        ("dec_depths", i32 * 4),
        ("ratio_min", C.c_double), ("ratio_max", C.c_double), ("pixels_min", C.c_double), ("pixels_max", C.c_double),
    ]


class Geometry(C.Structure):
    _fields_ = [
        ("pad_l", i32), ("pad_r", i32), ("pad_t", i32), ("pad_b", i32), ("padded_h", i32), ("padded_w", i32),
        ("net_h", i32), ("net_w", i32), ("gh", i32), ("gw", i32), ("factor", C.c_double),
    ]


class V1Geometry(C.Structure):
    _fields_ = [
        ("resized_h", i32), ("resized_w", i32), ("pad_l", i32), ("pad_r", i32), ("pad_t", i32), ("pad_b", i32),
        ("ratio", C.c_double),
    ]


class InferArgs(C.Structure):
    _fields_ = [
        ("rgb", vp), ("rgb_is_u8", i32), ("normalize", i32), ("B", i32), ("H", i32), ("W", i32),
        ("resolution_level", i32), ("camera_k", vp), ("camera_rays", vp), ("ray_scales", vp), ("workspace", vp),
        ("workspace_bytes", C.c_size_t),
        ("confidence", vp), ("intrinsics", vp), ("radius", vp), ("depth", vp), ("points", vp), ("rays", vp),
        ("depth_features", vp),
    ]


class V1Preprocess(C.Structure):
    _fields_ = [
        ("rgb", vp), ("rgb_is_u8", i32), ("scale255", i32), ("normalize", i32), ("B", i32), ("H", i32), ("W", i32),
        ("rh", i32), ("rw", i32), ("pad_l", i32), ("pad_t", i32), ("net_h", i32), ("net_w", i32), ("patches", vp),
    ]


class LayerNormAny(C.Structure):
    _fields_ = [
        ("inp", vp), ("in_f32", i32), ("out", vp), ("out_f32", i32), ("weight", vp), ("bias", vp),
        ("rows", i64), ("dim", i32), ("ld_in", i64), ("ld_out", i64), ("eps", f32), ("add", vp), ("add_mod", i64),
        ("s2d_h", i32), ("s2d_w", i32),
    ]


class V1Rays(C.Structure):
    _fields_ = [
        ("intr4", vp), ("B", i32), ("net_h", i32), ("net_w", i32), ("gh", i32), ("gw", i32),
        ("ln_w", vp), ("ln_b", vp), ("out", vp), ("sh_k", f32 * 81),
    ]


class V1Postprocess(C.Structure):
    _fields_ = [
        ("mean", vp), ("k4", vp), ("B", i32), ("net_h", i32), ("net_w", i32), ("pad_l", i32), ("pad_r", i32),
        ("pad_t", i32), ("pad_b", i32), ("H", i32), ("W", i32), ("out_depth", vp), ("out_points", vp),
    ]


class V1Config(C.Structure):
    _fields_ = [
        ("depths", i32 * 4), ("dims", i32 * 4), ("hidden", i32), ("heads", i32), ("expansion", i32),
        ("dec_depths", i32 * 3), ("net_h", i32), ("net_w", i32),
    ]


class InferV1Args(C.Structure):
    _fields_ = [
        ("rgb", vp), ("rgb_is_u8", i32), ("scale255", i32), ("normalize", i32), ("B", i32), ("H", i32), ("W", i32),
        ("intrinsics", vp), ("skip_camera", i32), ("workspace", vp), ("workspace_bytes", C.c_size_t),
        ("out_intrinsics", vp), ("out_points", vp), ("out_depth", vp),
    ]


class ProfileEntry(C.Structure):
    _fields_ = [("name", C.c_char * 48), ("ms", f32), ("flops", C.c_double), ("bytes", C.c_double)]


DT_F16, DT_F32 = 0, 1

EXPORTS = {
    "udb_version": (i32, []),
    "udb_last_error": (C.c_char_p, []),
    "udb_launch_count": (i64, []),
    "udb_profile_begin": (i32, [vp]),
    "udb_profile_end": (i32, [C.POINTER(ProfileEntry), i32]),
    "udb_gemm_f16": (i32, [C.POINTER(Gemm), vp]),
    "udb_conv3x3_halo_f16": (i32, [C.POINTER(ConvHalo), vp]),
    "udb_attention_f16": (i32, [C.POINTER(Attn), vp]),
    "udb_layernorm": (i32, [C.POINTER(LayerNorm), vp]),
    "udb_preprocess_patchify": (i32, [C.POINTER(Preprocess), vp]),
    "udb_posembed_bicubic": (i32, [vp, i32, i32, vp, i32, i32, vp]),
    "udb_set_cls_rows": (i32, [vp, vp, vp, i32, i32, i32, vp]),
    "udb_set_cls_rows_ln": (i32, [vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, vp]),
    "udb_small_linear_f32": (i32, [C.POINTER(SmallLinear), vp]),
    "udb_camera_attn4_f32": (i32, [vp, vp, vp, vp, i32, i32, i32, vp]),
    "udb_camera_intrinsics": (i32, [vp, i32, i32, i32, f32, i32, i32, vp, vp, vp, vp]),
    "udb_ray_embed": (i32, [C.POINTER(RayEmbed), vp]),
    "udb_upsample2x_nhwc_f16": (i32, [vp, vp, i32, i32, i32, i32, vp]),
    "udb_resize_ac_pad_nhwc_f16": (i32, [vp, vp, i32, i32, i32, i32, i32, i32, i32, vp]),
    "udb_reflect_pad1_nhwc_f16": (i32, [vp, vp, i32, i32, i32, i32, vp]),
    "udb_reflect_border_fill_nhwc_f16": (i32, [vp, i32, i32, i32, i32, vp]),
    "udb_postprocess": (i32, [C.POINTER(Postprocess), vp]),
    "udb_camera_adjust_k": (i32, [vp, i32, f32, i32, i32, vp, vp]),
    "udb_create": (i32, [C.POINTER(Config), C.POINTER(vp)]),
    "udb_destroy": (None, [vp]),
    "udb_set_weight": (i32, [vp, C.c_char_p, vp, C.POINTER(i64), i32, i32]),
    "udb_set_scalar": (i32, [vp, C.c_char_p, C.c_double]),
    "udb_geometry": (i32, [vp, i32, i32, i32, C.POINTER(Geometry)]),
    "udb_workspace_bytes": (C.c_size_t, [vp, i32, i32, i32, i32]),
    "udb_schedule_bytes": (C.c_size_t, [vp, i32, i32, i32, i32]),
    "udb_infer_v2": (i32, [vp, C.POINTER(InferArgs), vp]),
    # UniDepthV1 operators + engine
    "udb_v1_preprocess": (i32, [C.POINTER(V1Preprocess), vp]),
    "udb_v1_preprocess_vit": (i32, [C.POINTER(V1Preprocess), vp]),
    "udb_vit_tap_f16": (i32, [vp, vp, vp, i32, i32, i32, i32, vp]),
    "udb_layernorm_any": (i32, [C.POINTER(LayerNormAny), vp]),
    "udb_dwconv7_nhwc_f16": (i32, [vp, vp, vp, vp, i32, i32, i32, i32, vp]),
    "udb_max_accum_f16": (i32, [vp, vp, i64, i32, vp]),
    "udb_spatial_mean_f32": (i32, [vp, vp, i32, i32, i32, vp]),
    "udb_aa_resize_nhwc_f16": (i32, [vp, vp, i32, i32, i32, i32, i32, i32, vp]),
    "udb_v1_rays_sh81": (i32, [C.POINTER(V1Rays), vp]),
    "udb_v1_camera_intrinsics": (i32, [vp, vp, i32, i32, i32, f32, i32, i32, i32, vp, vp, vp, vp]),
    "udb_cross_attn_small": (i32, [vp, vp, vp, vp, vp, i32, i32, i32, i32, f32, vp]),
    "udb_softmax_rows": (i32, [vp, vp, i64, i32, i32, i32, f32, vp]),
    "udb_add_f32": (i32, [vp, vp, vp, vp, i64, vp]),
    "udb_copy_rows_f32_to_f16": (i32, [vp, vp, i32, i32, i32, i64, i64, vp]),
    "udb_conv3x3_c1_exp": (i32, [vp, vp, f32, vp, i32, i32, i32, i32, vp]),
    "udb_nystrom_landmarks": (i32, [vp, i32, vp, i32, vp, i32, i32, i32, vp]),
    "udb_nystrom_k2_pinv": (i32, [vp, vp, vp, vp, i32, i32, i32, vp]),
    "udb_nystrom_zk3": (i32, [vp, vp, i32, vp, i32, i32, i32, vp]),
    "udb_v1_mean_maps": (i32, [vp, vp, vp, vp, i32, i32, i32, i32, i32, vp]),
    "udb_v1_postprocess": (i32, [C.POINTER(V1Postprocess), vp]),
    "udb_v1_create": (i32, [C.POINTER(V1Config), C.POINTER(vp)]),
    "udb_v1_create_vit": (i32, [C.POINTER(V1Config), i32, C.POINTER(vp)]),
    "udb_v1_destroy": (None, [vp]),
    "udb_v1_set_weight": (i32, [vp, C.c_char_p, vp, C.POINTER(i64), i32, i32]),
    "udb_v1_set_scalar": (i32, [vp, C.c_char_p, C.c_double]),
    "udb_v1_geometry": (i32, [i32, i32, i32, i32, C.POINTER(V1Geometry)]),
    "udb_v1_workspace_bytes": (C.c_size_t, [vp, i32, i32, i32]),
    "udb_infer_v1": (i32, [vp, C.POINTER(InferV1Args), vp]),
    # peer-memory plumbing (multi-GPU gather)
    "udb_p2p_alloc": (i32, [C.c_size_t, C.POINTER(vp), vp]),
    "udb_p2p_open": (i32, [vp, C.POINTER(vp)]),
    "udb_p2p_close": (i32, [vp]),
    "udb_p2p_free": (i32, [vp]),
    "udb_p2p_barrier": (i32, [vp, vp, i32, i32, C.c_uint32, vp, vp]),
    "udb_p2p_copy": (i32, [vp, vp, C.c_size_t, vp]),
}

_lib = None


def lib():
    """Load libudb.so (built by unidepth_b200.build).  Raises if it is missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} not found: build the CUDA extension first (python -m unidepth_b200.build). "
                "unidepth_b200 has no CPU / PyTorch fallback.")
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in EXPORTS.items():
            if "UDB_LIB" in os.environ and not hasattr(l, name):
                continue      # experiment builds of older sources may lack newer entry points
            fn = getattr(l, name)
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def check(rc: int, what: str):
    if rc != 0:
        raise RuntimeError(f"{what} failed: {lib().udb_last_error().decode()}")


def profile(fn, stream_ptr, cap: int = 4096):
    """Run fn() between udb_profile_begin / udb_profile_end on the given stream; returns [(kernel, ms, flops, bytes)]."""
    l = lib()
    check(l.udb_profile_begin(stream_ptr), "udb_profile_begin")
    try:
        fn()
    finally:
        buf = (ProfileEntry * cap)()
        n = l.udb_profile_end(buf, cap)
    if n < 0:
        raise RuntimeError(f"udb_profile_end failed: {l.udb_last_error().decode()}")
    return [(buf[i].name.decode(), buf[i].ms, buf[i].flops, buf[i].bytes) for i in range(min(n, cap))]


def launch_count() -> int:
    return int(lib().udb_launch_count())
