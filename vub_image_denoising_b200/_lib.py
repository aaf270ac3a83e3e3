"""ctypes binding of libb200dn.so — the C ABI declared in include/b200dn.h.

There is exactly one compute path: the CUDA library.  If it has not been built, or a call fails, this
module raises; nothing here (or anywhere in the package) falls back to PyTorch/CPU math.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

PKG_DIR = Path(__file__).resolve().parent
# B200DN_LIB: load a diagnostics build of the same sources instead (python -m vub_image_denoising_b200._build --timeline)
LIB_PATH = Path(os.environ["B200DN_LIB"]) if os.environ.get("B200DN_LIB") else PKG_DIR / "libb200dn.so"

ABI_VERSION = 2

# enums (mirror include/b200dn.h)
PREC_BF16, PREC_FP16, PREC_BF16X2, PREC_BF16X3, PREC_FP16X2 = 0, 1, 2, 3, 4
PREC_NAMES = {"bf16": PREC_BF16, "fp16": PREC_FP16, "bf16x2": PREC_BF16X2, "bf16x3": PREC_BF16X3,
              "fp16x2": PREC_FP16X2, "fp32": PREC_BF16X3}
TWO_PLANE_PRECS = (PREC_BF16X2, PREC_BF16X3, PREC_FP16X2)
FP16_PRECS = (PREC_FP16, PREC_FP16X2)
MODE_CONV3X3, MODE_DOWN2X2, MODE_UP2X2, MODE_CONV1X1 = 0, 1, 2, 3
OUT_NHWC16, OUT_NCHW32 = 0, 1

# every symbol include/b200dn.h declares (tests check the .so exports exactly these)
EXPORTS = (
    "b200dn_last_error", "b200dn_abi_version", "b200dn_sm_count",
    "b200dn_pack_conv_weight", "b200dn_pack_convt_weight", "b200dn_packed_weight_bytes",
    "b200dn_igemm", "b200dn_igemm_plan", "b200dn_igemm_prepare", "b200dn_igemm_rebind_nchw", "b200dn_igemm_launch",
    "b200dn_igemm_launch_list", "b200dn_igemm_release", "b200dn_conv_in",
    "b200dn_dense_block_weight_bytes", "b200dn_pack_dense_block_weights", "b200dn_dense_block_prepare",
    "b200dn_dense_block_set_epilogue_constants",
    "b200dn_conv_chain_workspace_bytes", "b200dn_conv_chain_prepare",
    "b200dn_sampler_step", "b200dn_lerp",
    "b200dn_psnr_sse", "b200dn_ssim", "b200dn_psnr_sse_workspace_bytes", "b200dn_ssim_workspace_bytes",
    "b200dn_ssim_window", "b200dn_ssim_window_workspace_bytes",
    "b200dn_welch_psd", "b200dn_welch_psd_workspace_bytes",
    "b200dn_patch_gather_image", "b200dn_patch_gather", "b200dn_maxpool3x3s2", "b200dn_lpips_head",
    "b200dn_lpips_head_workspace_bytes",
    "b200dn_gauss_noise_u8", "b200dn_philox_normal", "b200dn_u8_to_norm", "b200dn_norm_to_u8",
)


class IgemmArgs(C.Structure):
    """struct b200dn_igemm_args"""
    _fields_ = [
        ("mode", C.c_int32), ("prec", C.c_int32),
        ("B", C.c_int32), ("H", C.c_int32), ("W", C.c_int32),
        ("cin", C.c_int32), ("cout", C.c_int32),
        ("in_", C.c_void_p * 2), ("in_ctot", C.c_int32),
        ("wpacked", C.c_void_p), ("bias", C.c_void_p), ("slope", C.c_void_p),
        ("out_kind", C.c_int32),
        ("out", C.c_void_p * 2), ("out_ctot", C.c_int32), ("out_coff", C.c_int32),
        ("res", C.c_void_p * 2), ("res_ctot", C.c_int32),
        ("out_nchw", C.c_void_p), ("res_nchw", C.c_void_p), ("res_bmod", C.c_int32),
        ("block_n", C.c_int32), ("max_ctas", C.c_int32), ("m_tiles", C.c_int32), ("impl", C.c_int32),
        ("sat_flag", C.c_void_p),
    ]


class DenseBlockArgs(C.Structure):
    """struct b200dn_dense_block_args"""
    _fields_ = [
        ("prec", C.c_int32), ("B", C.c_int32), ("H", C.c_int32), ("W", C.c_int32), ("channels", C.c_int32),
        ("in_", C.c_void_p), ("in_ctot", C.c_int32),
        ("out", C.c_void_p), ("out_ctot", C.c_int32), ("out_coff", C.c_int32),
        ("wfused", C.c_void_p), ("bias", C.c_void_p * 4), ("slope", C.c_void_p * 4),
        ("max_ctas", C.c_int32), ("sat_flag", C.c_void_p), ("timeline", C.c_void_p),
    ]


class IgemmPlanInfo(C.Structure):
    """struct b200dn_igemm_plan_info"""
    _fields_ = [(n, C.c_int32) for n in (
        "kernel", "mt", "block_n", "num_n_tiles", "num_tiles", "grid", "wres", "num_slabs", "slab_bytes", "num_stages",
        "stage_bytes", "w_taps", "tmem_cols", "epi_staged", "data_bytes_used", "data_bytes_budget")]


class LpipsTap(C.Structure):
    """struct b200dn_lpips_tap"""
    _fields_ = [("feat", C.c_void_p * 2), ("weight", C.c_void_p), ("H", C.c_int32), ("W", C.c_int32), ("C", C.c_int32)]


SSIM_MAX_RADIUS = 15                     # B200DN_SSIM_MAX_RADIUS


class SsimWindowOpts(C.Structure):
    """struct b200dn_ssim_window_opts"""
    _fields_ = [("radius", C.c_int32), ("win_size", C.c_int32), ("cov_norm", C.c_float), ("C1", C.c_float),
                ("C2", C.c_float), ("weights", C.c_float * (2 * SSIM_MAX_RADIUS + 1))]


E_ARG, E_CUDA, E_UNSUP = -1, -2, -3      # B200DN_E_*

_lib = None


def lib_available() -> bool:
    return LIB_PATH.exists()


def _check_fresh() -> None:
    """The .so is git-ignored and travels with the snapshot: refuse to run against a binary whose recorded source
    digest (build/sources.sha256, written by _build.build_lib) no longer matches csrc/ + include/b200dn.h, so that GPU
    parity results always reflect the sources at HEAD.  B200DN_ALLOW_STALE=1 skips the check."""
    if os.environ.get("B200DN_ALLOW_STALE") == "1" or os.environ.get("B200DN_LIB"):
        return
    from . import _build
    if _build.STAMP.exists() and _build.STAMP.read_text().strip() != _build._digest():
        raise RuntimeError(
            f"{LIB_PATH} is stale: csrc/ or include/b200dn.h changed since it was built.  Rebuild it with "
            "`python -m vub_image_denoising_b200._build` (or __graft_entry__.build()).")


def lib() -> C.CDLL:
    """Load (once) and return the library.  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -m vub_image_denoising_b200._build` "
            "(or __graft_entry__.build()).  There is no fallback path.")
    _check_fresh()
    L = C.CDLL(str(LIB_PATH))
    vp, i32, i64, f32 = C.c_void_p, C.c_int, C.c_int64, C.c_float
    L.b200dn_last_error.restype = C.c_char_p
    L.b200dn_last_error.argtypes = []
    L.b200dn_abi_version.restype = i32
    L.b200dn_sm_count.restype = i32
    L.b200dn_packed_weight_bytes.restype = i64
    L.b200dn_packed_weight_bytes.argtypes = [i32, i32, i32, i32]
    L.b200dn_pack_conv_weight.argtypes = [vp, i32, i32, i32, i32, i32, vp, vp]
    L.b200dn_pack_convt_weight.argtypes = [vp, i32, i32, i32, vp, vp]
    L.b200dn_igemm.argtypes = [C.POINTER(IgemmArgs), vp]
    L.b200dn_igemm_plan.argtypes = [C.POINTER(IgemmArgs), i32, C.POINTER(IgemmPlanInfo)]
    L.b200dn_igemm_prepare.argtypes = [C.POINTER(IgemmArgs), C.POINTER(vp)]
    L.b200dn_igemm_rebind_nchw.argtypes = [vp, vp, vp, i32]
    L.b200dn_igemm_launch.argtypes = [vp, vp]
    L.b200dn_igemm_launch_list.argtypes = [C.POINTER(vp), i32, vp]
    L.b200dn_igemm_release.argtypes = [vp]
    L.b200dn_igemm_release.restype = None
    L.b200dn_dense_block_weight_bytes.restype = i64
    L.b200dn_dense_block_weight_bytes.argtypes = [i32]
    L.b200dn_pack_dense_block_weights.argtypes = [vp, vp, vp, vp, i32, i32, vp, vp]
    L.b200dn_dense_block_prepare.argtypes = [C.POINTER(DenseBlockArgs), C.POINTER(vp)]
    L.b200dn_dense_block_set_epilogue_constants.argtypes = [vp, C.POINTER(C.POINTER(C.c_float)), C.POINTER(C.POINTER(C.c_float))]
    L.b200dn_conv_chain_workspace_bytes.restype = i64
    L.b200dn_conv_chain_workspace_bytes.argtypes = [C.POINTER(IgemmArgs), i32]
    L.b200dn_conv_chain_prepare.argtypes = [C.POINTER(IgemmArgs), i32, vp, i32, C.POINTER(vp)]
    L.b200dn_conv_in.argtypes = [vp, i32, i32, vp, i64, i64, i64, i32, i32, i32, i32, vp, vp, vp, i32, vp, vp, i32, vp, vp]
    L.b200dn_sampler_step.argtypes = [vp, vp, vp, vp, f32, f32, f32, f32, vp, i64, vp]
    L.b200dn_lerp.argtypes = [vp, vp, f32, f32, vp, i64, vp]
    L.b200dn_psnr_sse.argtypes = [vp, vp, i64, i64, vp, vp, i64, vp]
    L.b200dn_ssim.argtypes = [vp, vp, i64, i32, i32, f32, vp, vp, i64, vp]
    L.b200dn_psnr_sse_workspace_bytes.restype = i64
    L.b200dn_psnr_sse_workspace_bytes.argtypes = [i64, i64]
    L.b200dn_ssim_workspace_bytes.restype = i64
    L.b200dn_ssim_workspace_bytes.argtypes = [i64, i32, i32]
    L.b200dn_ssim_window.argtypes = [vp, vp, i64, i32, i32, C.POINTER(SsimWindowOpts), vp, vp, vp, i64, vp]
    L.b200dn_ssim_window_workspace_bytes.restype = i64
    L.b200dn_ssim_window_workspace_bytes.argtypes = [i64, i32, i32]
    L.b200dn_welch_psd.argtypes = [vp, i64, i64, vp, vp, i64, vp]
    L.b200dn_welch_psd_workspace_bytes.restype = i64
    L.b200dn_welch_psd_workspace_bytes.argtypes = [i64, i64]
    L.b200dn_patch_gather_image.argtypes = [vp, vp, i32, i32, i32, i32, vp, vp, i32, i32, i32, i32, i32, i32, i32, vp,
                                            vp, vp]
    L.b200dn_patch_gather.argtypes = [vp, vp, i32, i32, i32, i32, i32, i32, i32, i32, i32, i32, vp, vp, vp]
    L.b200dn_maxpool3x3s2.argtypes = [vp, vp, i32, i32, i32, i32, i32, vp, vp, vp]
    L.b200dn_lpips_head_workspace_bytes.restype = i64
    L.b200dn_lpips_head_workspace_bytes.argtypes = [C.POINTER(LpipsTap), i32, i32]
    L.b200dn_lpips_head.argtypes = [C.POINTER(LpipsTap), i32, i32, i32, vp, vp, i64, vp]
    L.b200dn_gauss_noise_u8.argtypes = [vp, i32, i32, i32, i32, vp, C.c_uint64, C.c_uint32, vp, vp, vp, vp]
    L.b200dn_philox_normal.argtypes = [vp, i64, C.c_uint64, C.c_uint32, vp]
    L.b200dn_u8_to_norm.argtypes = [vp, i32, i32, i32, i32, vp, vp]
    L.b200dn_norm_to_u8.argtypes = [vp, i32, i32, i32, i32, vp, vp]
    for name in EXPORTS:
        fn = getattr(L, name)
        if name not in ("b200dn_last_error", "b200dn_packed_weight_bytes", "b200dn_igemm_release",
                        "b200dn_psnr_sse_workspace_bytes", "b200dn_ssim_workspace_bytes",
                        "b200dn_ssim_window_workspace_bytes",
                        "b200dn_welch_psd_workspace_bytes", "b200dn_dense_block_weight_bytes",
                        "b200dn_conv_chain_workspace_bytes", "b200dn_lpips_head_workspace_bytes"):
            fn.restype = i32
    if L.b200dn_abi_version() != ABI_VERSION:
        raise RuntimeError("libb200dn.so ABI version mismatch; rebuild the library")
    _lib = L
    return L


def check(rc: int, what: str = "") -> None:
    """Raise RuntimeError (the reference surfaces shape/device errors as RuntimeError too) on rc < 0."""
    if rc < 0:
        msg = lib().b200dn_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"libb200dn {what} failed (code {rc}): {msg}")
