"""ctypes binding of libmri_b200.so (the C ABI declared in include/mri_b200.h).

The library is the product: there is no Python/torch fallback for any kernel.  If the shared
object is missing or the device is not a compute-capability-10.x GPU, calls fail loudly.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmri_b200.so")
if os.environ.get("MRI_B200_LIB"):   # kernel-probe builds (tools/): an explicitly named library
    LIB_PATH = os.environ["MRI_B200_LIB"]


class MriGemmArgs(C.Structure):
    _fields_ = [
        ("a_maps", C.c_void_p),
        ("b_map", C.c_void_p),
        ("o_maps", C.c_void_p),
        ("ktable", C.c_void_p),
        ("n_kb", C.c_int32),
        ("n_class", C.c_int32),
        ("tiles", C.c_int32 * 4),
        ("box", C.c_int32 * 4),
        ("ext", C.c_int32 * 4),
        ("n_tiles_n", C.c_int32),
        ("block_n", C.c_int32),
        ("n_total", C.c_int32),
        ("bz_sel", C.c_int32 * 2),
        ("sample_dim", C.c_int32),
        ("out_f32", C.c_int32),
        ("bias", C.c_void_p),
        ("bias_m", C.c_void_p),
        ("rowbias", C.c_void_p),
        ("rowbias_ld", C.c_int32),
        ("stats", C.c_void_p),
        ("stats_ld", C.c_int32),
        ("stats_cpg", C.c_int32),
        ("stages", C.c_int32),
        ("sched", C.c_int32),
        ("r_maps", C.c_void_p),
        ("r_base", C.c_void_p),
        ("r_cls_off", C.c_int64 * 8),
        ("r_stride", C.c_int64 * 4),
        ("sk_partials", C.c_void_p),
        ("sk_flags", C.c_void_p),
        ("sk_ctas", C.c_int32),
        ("swap_ab", C.c_int32),
        ("staging2", C.c_int32),
        ("xreuse", C.c_int32),
        ("tile_fast_dim", C.c_int32),
        ("trace", C.c_void_p),
    ]


class MriWgradArgs(C.Structure):
    _fields_ = [
        ("a_maps", C.c_void_p),
        ("dy_maps", C.c_void_p),
        ("ktable", C.c_void_p),
        ("n_kb", C.c_int32),
        ("n_class", C.c_int32),
        ("tiles", C.c_int32 * 4),
        ("box", C.c_int32 * 4),
        ("n_total", C.c_int32),
        ("co_blocks", C.c_int32),
        ("splits", C.c_int32),
        ("group", C.c_int32),
        ("dw", C.c_void_p),
        ("dw_rows", C.c_int32),
        ("dw_ld", C.c_int32),
        ("stages", C.c_int32),
        ("xgroup", C.c_int32),
    ]


class MriAttnArgs(C.Structure):
    _fields_ = [("qk_map", C.c_void_p), ("vt_map", C.c_void_p), ("out", C.c_void_p),
                ("batch", C.c_int32), ("heads", C.c_int32), ("n", C.c_int32), ("d", C.c_int32),
                ("C", C.c_int32), ("k_col0", C.c_int32), ("v_row0", C.c_int32), ("ld_out", C.c_int32),
                ("scale", C.c_float), ("reserved", C.c_int32)]


class MriGatherSeg(C.Structure):
    _fields_ = [
        ("dst", C.c_void_p),
        ("idx", C.c_void_p),
        ("src", C.c_void_p * 4),
        ("n", C.c_int64),
        ("block0", C.c_int64),
        ("dst_bf16", C.c_int32),
        ("reserved", C.c_int32),
    ]


class MriAdamSeg(C.Structure):
    _fields_ = [("p", C.c_void_p), ("g", C.c_void_p), ("m", C.c_void_p), ("v", C.c_void_p),
                ("n", C.c_int64), ("block0", C.c_int64)]


class MriEmaSeg(C.Structure):
    _fields_ = [("e", C.c_void_p), ("p", C.c_void_p), ("n", C.c_int64), ("block0", C.c_int64)]


class MriFinalSeg(C.Structure):
    _fields_ = [("dst", C.c_void_p), ("src", C.c_void_p), ("idx", C.c_void_p), ("n", C.c_int64),
                ("block0", C.c_int64), ("batch", C.c_int32), ("ld", C.c_int32)]


# name -> (restype, argtypes); mirrors include/mri_b200.h one to one
_vp, _i, _i64, _f, _u64 = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_uint64
SIGNATURES = {
    "mri_abi_version": (_i, []),
    "mri_last_error": (C.c_char_p, []),
    "mri_device_ok": (_i, []),
    "mri_tmap_encode": (_i, [_vp, _u64, _i, _i, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64),
                             C.POINTER(C.c_uint32), _i]),
    "mri_gemm_smem_bytes": (_i, [_i, _i, _i]),
    "mri_gemm_launch": (_i, [C.POINTER(MriGemmArgs), _vp]),
    "mri_gemm_workspace_bytes": (_i, [C.POINTER(C.c_int)]),
    "mri_gn_stats": (_i, [_vp, _vp, _i, _i64, _i, _i, _i, _i, _vp]),
    "mri_gn_apply": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _i, _i64, _i, _i, _i, _i, _i, _f,
                          _i, _vp]),
    "mri_sinusoidal": (_i, [_vp, _vp, _vp, _i, _i, _vp]),
    "mri_linear": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    "mri_im2col": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "mri_adam_step": (_i, [_vp, _i, _i64, _f, _f, _f, _f, _f, _vp, _vp, _vp, _vp]),
    "mri_ema_update": (_i, [_vp, _i, _i64, C.c_double, _i, _vp, _vp, _vp]),
    "mri_gather_pack": (_i, [_vp, _i, _i64, _vp]),
    "mri_grad_finalize": (_i, [_vp, _i, _i64, _vp]),
    "mri_im2col4": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "mri_tap_gather": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "mri_nhwc_to_nchw": (_i, [_vp, _vp, _i, _i64, _i, _i, _vp]),
    "mri_nchw_to_nhwc": (_i, [_vp, _vp, _i, _i64, _i, _i, _vp]),
    "mri_attn_flash_supported": (_i, [_i]),
    "mri_attn_flash_launch": (_i, [C.POINTER(MriAttnArgs), _vp]),
    "mri_softmax_rows": (_i, [_vp, _vp, _i64, _i, _i, _i, _f, _vp]),
    "mri_thin_in_conv": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "mri_copy_cast": (_i, [_vp, _i, C.POINTER(C.c_int64), _vp, _i, C.POINTER(C.c_int64),
                           C.POINTER(C.c_int64), _vp]),
    "mri_memset_zero": (_i, [_vp, _i64, _vp]),
    "mri_masked_stats": (_i, [_vp, _i, _i64, _i64, _i64, _i64, _i64, _f, _vp, _vp, _vp]),
    "mri_slice_normalize_resize": (_i, [_vp, _i, _i64, _i, _i, _i64, _i64, _vp, _i, _i, _vp, _i64,
                                        _vp]),
    "mri_volume_normalize_patch": (_i, [_vp, _i, _i, _i, _i64, _i64, _i64, _vp, _f, _i, _i, _i, _i,
                                        _i, _i, _vp, _vp]),
    "mri_q_sample": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i64, _vp]),
    "mri_ddpm_step": (_i, [_vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i64, _vp]),
    "mri_ddim_step": (_i, [_vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _i, _i64, _vp]),
    "mri_dpmpp_step": (_i, [_vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _i, _i64, _vp]),
    "mri_step_table_advance": (_i, [_vp, _i, _vp, _vp, _i, _vp]),
    "mri_inpaint_merge": (_i, [_vp, _vp, _vp, _vp, _vp, _u64, _vp, _i64, _vp, _vp, _i, _i64, _vp]),
    "mri_kspace_work_bytes": (_i, [_i, _i, _i, _i, _vp]),
    "mri_kspace_merge": (_i, [_vp, _vp, _vp, _vp, _vp, _u64, _vp, _i64, _vp, _vp, _vp, C.c_size_t, _i,
                              _i, _i, _i, _vp]),
    "mri_kspace3d_work_bytes": (_i, [_i, _i, _i, _i, _i, _vp]),
    "mri_dc_project3d": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, C.c_size_t, _i, _i, _i, _i, _i, _vp]),
    "mri_dc_mask": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, C.c_size_t, _i, _i64, _vp]),
    "mri_guided_x0": (_i, [_vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _i, _i64, _vp]),
    "mri_guided_eps": (_i, [_vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i64, _vp]),
    "mri_repaint_undo": (_i, [_vp, _vp, _vp, _u64, _vp, _vp, _vp, _i, _i64, _vp]),
    "mri_vb_terms": (_i, [_vp, _vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _vp, _i,
                          _i, _i64, _vp]),
    "mri_minsnr_loss": (_i, [_vp, _vp, _vp, _vp, _f, _vp, _vp, _i, _i64, _vp]),
    "mri_add_i64": (_i, [_vp, _i, _i64, _vp]),
    "mri_randn_offset_increment": (_i, [_i64, C.POINTER(C.c_uint64)]),
    "mri_rng_seed": (_i, [_vp, _u64, _u64, _vp]),
    "mri_randn": (_i, [_vp, _i64, _vp, _vp]),
    "mri_q_sample_rng": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i64, _vp]),
    "mri_ddpm_step_rng": (_i, [_vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i64, _vp]),
    "mri_step_advance": (_i, [_vp, _vp, _i, _i64, _vp, _u64, _vp]),
    "mri_tap_gather_step": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _i, _i, _vp, _vp, _vp,
                                 _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "mri_wgrad_launch": (_i, [C.POINTER(MriWgradArgs), _vp]),
    "mri_gn_bwd_reduce": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i64, _i, _i, _i, _i, _f, _i, _vp]),
    "mri_gn_bwd_apply": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i64, _i, _i, _i, _i, _f,
                              _i, _vp, _vp]),
    "mri_add_bf16": (_i, [_vp, _vp, _vp, _i64, _vp]),
    "mri_gn_split": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _i, _i64, _i, _i, _i, _i, _f, _i, _vp]),
    "mri_stats_f32": (_i, [_vp, _vp, _i, _i64, _i, _i, _vp]),
    "mri_split3": (_i, [_vp, _vp, _i64, _i, _i, _i64, _i64, _i64, _i64, _i, _i, _vp]),
    "mri_softmax_rows_split": (_i, [_vp, _vp, _i64, _i, _i, _i, _i, _f, _vp]),
    "mri_bf16_residual_nchw": (_i, [_vp, _vp, _i, _i64, _i64, _vp]),
    "mri_copy_window_nhwc": (_i, [_vp, _vp, _vp] + [_i] * 12 + [_vp]),
    "mri_resize_bilinear_nhwc": (_i, [_vp, _vp] + [_i] * 6 + [_vp]),
    "mri_resize_bilinear_nhwc_bwd": (_i, [_vp, _vp, _vp] + [_i] * 6 + [_vp]),
    "mri_softmax_bwd": (_i, [_vp, _vp, _vp, _i64, _i, _i, _i, _f, _vp]),
    "mri_linear_bwd": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp]),
    "mri_silu": (_i, [_vp, _vp, _i64, _vp]),
    "mri_silu_bwd": (_i, [_vp, _vp, _vp, _i64, _vp]),
    "mri_minsnr_loss_bwd": (_i, [_vp, _vp, _vp, _vp, _f, _vp, _vp, _i, _i64, _vp]),
}


class MriError(RuntimeError):
    pass


_lib: Optional[C.CDLL] = None


def load() -> C.CDLL:
    """Load libmri_b200.so (built by `make -C mri_image_generation_b200/csrc` or
    __graft_entry__.build()).  Raises if it is missing: no fallback exists."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise MriError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; "
            "g.build()'` (nvcc, sm_100a).  This package has no CPU or PyTorch fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    if lib.mri_abi_version() != 1:
        raise MriError("libmri_b200.so ABI version mismatch")
    _lib = lib
    return lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load().mri_last_error().decode("utf-8", "replace")
        raise MriError(f"{what or 'libmri_b200'} failed (rc={rc}): {msg}")


def current_stream_ptr() -> int:
    import torch

    return torch.cuda.current_stream().cuda_stream


def require_device() -> None:
    """Fail loudly unless a Blackwell (CC 10.x) GPU is current."""
    import torch

    if not torch.cuda.is_available():
        raise MriError("mri_image_generation_b200 needs a B200 GPU (CUDA not available); "
                       "there is no CPU path")
    rc = load().mri_device_ok()
    if rc != 1:
        raise MriError("mri_image_generation_b200 kernels are built for sm_100a only "
                       f"(mri_device_ok() = {rc})")
