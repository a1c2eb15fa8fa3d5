"""ctypes binding of libextdm_b200.so (the C ABI declared in include/extdm_b200.h).

The library is built in-tree by build.py (nvcc, sm_100a).  There is NO fallback: if the shared object is
missing or a kernel launch fails, the caller gets an exception.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("EXTDM_LIB") or os.path.join(_HERE, "libextdm_b200.so")    # EXTDM_LIB: A/B builds (build.py)


class ExtdmGemm(C.Structure):
    """Mirror of `struct ExtdmGemm` (include/extdm_b200.h)."""
    _fields_ = [
        ("a0", C.c_void_p), ("a1", C.c_void_p),
        ("a0_channels", C.c_int), ("a1_channels", C.c_int),
        ("a0_dim", C.c_longlong * 4), ("a0_stride", C.c_longlong * 4),
        ("a1_dim", C.c_longlong * 4), ("a1_stride", C.c_longlong * 4),
        ("box", C.c_int * 4), ("start", C.c_int * 4), ("count", C.c_int * 4),
        ("ntaps", C.c_int), ("tap", (C.c_byte * 4) * 64),
        ("w", C.c_void_p), ("n", C.c_int), ("w_rows", C.c_int),
        ("out", C.c_void_p), ("out_fp32", C.c_int), ("out_base", C.c_longlong),
        ("out_stride", C.c_longlong * 4), ("col_group", C.c_int), ("col_group_stride", C.c_longlong),
        ("bias", C.c_void_p),
        ("res", C.c_void_p), ("res_fp32", C.c_int), ("res_base", C.c_longlong), ("res_stride", C.c_longlong * 4),
        ("col_scale", C.c_void_p), ("col_shift", C.c_void_p),
        ("act", C.c_int), ("block_n", C.c_int),
        ("gn_partials", C.c_void_p),
        ("tf32", C.c_int),
        ("n_phase", C.c_int), ("phase_out_offset", C.c_longlong * 4),
    ]


_I, _L, _F, _P = C.c_int, C.c_longlong, C.c_float, C.c_void_p

# name -> argument ctypes (every function returns int status unless listed in _RET)
PROTOTYPES = {
    "extdm_abi_version": [],
    "extdm_last_error": [],
    "extdm_sizeof_gemm": [],
    "extdm_conv_gemm": [C.POINTER(ExtdmGemm), _P],
    "extdm_image_to_cl": [_P, _I, _I, _P, _I, _I, _P, _I, _I, _P, _I, _I, _I, _I, _P],
    "extdm_avgpool2_f32_cl": [_P, _P, _L, _I, _I, _I, _P],
    "extdm_upsample2_f32_cl": [_P, _P, _L, _I, _I, _I, _P],
    "extdm_region_moments": [_P, _I, _I, _I, _I, _I, _I, _F, _P, _P, _P],
    "extdm_pca_affine": [_P, _P, _I, _P],
    "extdm_sparse_motion": [_P, _I, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _F, _P, _I, _P, _P],
    "extdm_sparse_motion_src": [_P, _I, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _F, _P, _I, _P, _P],
    "extdm_flow_compose": [_P, _I, _P, _I, _I, _I, _I, _I, _P, _P, _P],
    "extdm_bg_head": [_P, _I, _I, _I, _P, _P, _I, _I, _P, _P],
    "extdm_groupnorm_stats": [_P, _P, _I, _L, _I, _I, _P],
    "extdm_groupnorm_apply": [_P, _P, _I, _P, _P, _P, _L, _I, _P, _P, _I, _L, _I, _I, _F, _P],
    "extdm_chan_layernorm": [_P, _L, _I, _P, _L, _I, _P, _P, _L, _L, _F, _P],
    "extdm_temporal_prenorm": [_P, _P, _P, _P, _P, _P, _L, _I, _F, _P],
    "extdm_adaptor_workspace_floats": [_I, _I],
    "extdm_adaptor_normalize": [_P, _L, _P, _P, _P, _I, _I, _I, _I, _F, _P],
    "extdm_space_to_depth": [_P, _P, _L, _I, _I, _I, _P],
    "extdm_im2col7_flow": [_P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _P],
    "extdm_im2col13x_flow": [_P, _P, _I, _I, _I, _I, _I, _I, _P],
    "extdm_init_corner_fix": [_P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _P],
    "extdm_upsample2_border": [_P, _P, _P, _P, _P, _L, _I, _I, _I, _P],
    "extdm_bilinear_resize_cl": [_P, _P, _L, _I, _I, _I, _I, _I, _P],
    "extdm_time_mlp": [_P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _P],
    "extdm_head_project": [_P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P],
    "extdm_head_project_gn": [_P] * 10 + [_I] + [_P] * 5 + [_I] * 6 + [_F, _P],
    "extdm_window_attention": [_P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _I, _I, _I, _P],
    "extdm_stw_fused_supported": [_I, _I, _I, _I, _I, _I],
    "extdm_stw_fused": [_P, _P, _P, _P, _P, _P, _P, _P, _P] + [_I] * 13 + [_F, _P],
    "extdm_stw_fused_pre_supported": [_I, _I, _I, _I, _I, _I],
    "extdm_stw_fused_pre": [_P] * 11 + [_I] * 13 + [_F, _P],
    "extdm_groupnorm_affine": [_P, _I, _P, _P, _P, _I, _L, _I, _I, _F, _P],
    "extdm_temporal_fused_supported": [_I, _I, _I, _I],
    "extdm_temporal_fused": [_P] * 10 + [_I] * 6 + [_F, _P],
    "extdm_cross_attention": [_P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _P],
    "extdm_maxpool2_frames_cl": [_P, _P, _I, _I, _L, _L, _I, _I, _I, _P],
    "extdm_bilinear_resize_frames_cl": [_P, _P, _I, _I, _L, _L, _I, _I, _I, _I, _I, _P],
    "extdm_temporal_attention": [_P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P],
    "extdm_ddim_threshold": [_P, _P, _F, _F, _F, _P, _I, _I, _P],
    "extdm_ddim_update": [_P, _P, _P, _P, _F, _F, _F, _F, _F, _P, _P, _I, _I, _P],
    "extdm_ddim_update_seeded": [_P, _P, _P, _I, _P, _F, _F, _F, _F, _F, _P, _P, _I, _I, _P],
    "extdm_ddpm_threshold": [_P, _P, _P, _P, _F, _P, _I, _I, _P],
    "extdm_ddpm_update": [_P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _P],
    "extdm_ddpm_fill_normal": [_P, _P, _I, _I, _P],
    "extdm_ddpm_broadcast_row": [_P, _P, _P, _I, _I, _P],
    "extdm_ddpm_advance": [_P, _P, _I, _P, _I, _P],
    "extdm_dpmpp_update": [_P, _P, _P, _P, _P, _I, _P, _F, _F, _F, _F, _F, _F, _I, _P, _P, _I, _I, _P],
    "extdm_q_sample": [_P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _P],
    "extdm_denoise_loss": [_P, _P, _P, _I, _I, _I, _I, _P],
    "extdm_q_interpolate": [_P, _P, _I, _P, _P, _P, _P, _F, _F, _P, _I, _I, _P],
    "extdm_impose_known": [_P, _P, _P, _P, _P, _F, _F, _I, _I, _P, _P, _I, _I, _I, _P],
    "extdm_warp_blend_cl": [_P, _P, _P, _P, _P, _L, _L, _I, _I, _I, _I, _I, _I, _P],
    "extdm_warp_image": [_P, _P, _I, _P, _P, _P, _P, _L, _L, _I, _I, _I, _I, _P],
    "extdm_warp_taps": [_P, _P, _P, _P, _P, _L, _I, _I, _I, _I, _P],
    "extdm_bn_relu_cl": [_P, _P, _P, _P, _L, _I, _P],
    "extdm_avgpool2_cl": [_P, _P, _L, _I, _I, _I, _P],
    "extdm_im2col7_image": [_P, _P, _L, _I, _I, _P],
    "extdm_ncthw_to_cl": [_P, _P, _I, _I, _L, _L, _P],
    "extdm_cl_to_ncthw": [_P, _P, _I, _I, _L, _L, _P],
}
_RET = {"extdm_last_error": C.c_char_p, "extdm_adaptor_workspace_floats": C.c_longlong}

ABI_VERSION = 5          # extdm_abi_version() of the library this binding mirrors (include/extdm_b200.h)
_lib = None


class ExtdmError(RuntimeError):
    pass


def load():
    """dlopen the in-tree library (no CUDA call is made by loading it)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ExtdmError(f"{LIB_PATH} not found: run __graft_entry__.build() / python build.py first "
                             "(there is no CPU or PyTorch fallback for the hot path)")
        lib = C.CDLL(LIB_PATH)
        for name, args in PROTOTYPES.items():
            fn = getattr(lib, name)
            fn.argtypes = args
            fn.restype = _RET.get(name, C.c_int)
        if lib.extdm_abi_version() != ABI_VERSION:
            raise ExtdmError(f"{LIB_PATH}: ABI version {lib.extdm_abi_version()}, this binding expects {ABI_VERSION} "
                             "(stale build? run build.py)")
        if lib.extdm_sizeof_gemm() != C.sizeof(ExtdmGemm):
            raise ExtdmError("struct ExtdmGemm: ctypes mirror and compiled library disagree on the layout")
        _lib = lib
    return _lib


_launches = 0


def launches():
    """Number of kernel-launching ABI calls made so far through call() (bench.py's gpu_launches)."""
    return _launches


def call(name, *args):
    global _launches
    lib = load()
    rc = getattr(lib, name)(*args)
    _launches += 1
    if rc != 0:
        raise ExtdmError(f"{name} failed ({rc}): {lib.extdm_last_error().decode()}")
