"""vub_image_denoising_b200 — B200-native (sm_100a) drop-in for the denoising hot path of
pierregab/VUB_Image_denoising: RDUNet / RDUNet_T forward, DiffusionModel.improved_sampling, on-device
noise synthesis, PSNR/SSIM and LPIPS.  All compute goes through libb200dn.so (include/b200dn.h); there is no
CPU or PyTorch fallback.
"""
from ._lib import lib, lib_available, LIB_PATH  # noqa: F401
from .rdunet import RDUNet, RDUNet_T, init_weights, ForwardPlan  # noqa: F401
from .diffusion import DiffusionModel  # noqa: F401
from . import metrics, noise, sharding, shim, ops, sidd, perceptual  # noqa: F401

__all__ = ["RDUNet", "RDUNet_T", "DiffusionModel", "init_weights", "ForwardPlan", "metrics", "noise",
           "sharding", "shim", "ops", "sidd", "perceptual", "lib", "lib_available", "LIB_PATH"]
__version__ = "0.1.0"
