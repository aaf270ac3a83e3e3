/*
 * b200dn.h — C ABI of the B200-native RDUNet denoising hot path (libb200dn.so).
 *
 * Every entry point enqueues work on the caller's CUDA stream (`stream` is a
 * cudaStream_t passed as void*), performs no hidden synchronisation, never
 * throws across the ABI, and returns 0 on success or a negative B200DN_E_* code
 * (text via b200dn_last_error()).  All pointers are raw device pointers unless
 * the name says "host".  There is no CPU fallback: on a machine without an
 * sm_100 GPU every compute call returns B200DN_E_CUDA.
 *
 * What each entry point replaces in the reference (pierregab/VUB_Image_denoising,
 * paths relative to the reference root):
 *
 *   b200dn_igemm            nn.Conv2d(.,.,3,padding=1)+nn.PReLU      UNet/RDUNet_model.py:61,74-75,86-87,98-101
 *                           torch.cat in the dense block (eliminated) UNet/RDUNet_model.py:107-115
 *                           `out_3 + x` dense residual               UNet/RDUNet_model.py:115
 *                           nn.Conv2d(C,2C,2,stride=2)+PReLU         UNet/RDUNet_model.py:49-56
 *                           nn.ConvTranspose2d(C,C,2,stride=2)+PReLU UNet/RDUNet_model.py:62,66-68
 *                           OutputBlock.conv_2 + `+ inputs`          UNet/RDUNet_model.py:83-93,186
 *   b200dn_igemm_prepare / _launch / _launch_list / _rebind_nchw / _release
 *                           the same layers as b200dn_igemm, with the launch configuration and the encoded tensor
 *                           maps kept in an opaque handle: the ~70 modules RDUNet.forward chains per call
 *                           (UNet/RDUNet_model.py:157-186) become one C call over a prebuilt list
 *   b200dn_dense_block_prepare / b200dn_pack_dense_block_weights
 *                           DenoisingBlock as one kernel             UNet/RDUNet_model.py:95-115
 *   b200dn_conv_chain_prepare / b200dn_conv_chain_workspace_bytes
 *                           conv_0..conv_3 of a DenoisingBlock of any width as ONE persistent launch whose tiles
 *                           wait on the tiles they read, not on a launch boundary   UNet/RDUNet_model.py:106-115
 *   b200dn_conv_in          InputBlock.conv_1 + actv_1, t-plane cat  UNet/RDUNet_model.py:71-81,
 *                                                                    diffusion_denoising/Unet/Unet_model.py:133-136
 *   b200dn_pack_conv_weight / b200dn_pack_convt_weight
 *                           state_dict layout -> kernel layout       (OIHW / IOHW fp32 -> [plane][tap][CoutPad][CinPad])
 *   b200dn_sampler_step     x_t - x_tilde + x_tilde_prev             diffusion_denoising/diffusion_RDUnet.py:45,48,49
 *   b200dn_lerp             forward_diffusion                        diffusion_denoising/diffusion_RDUnet.py:33-36
 *   b200dn_psnr_sse         calculate_psnr / peak_signal_noise_ratio evaluate_Unet_diffusion/evaluate_model.py:36-41,
 *                                                                    evaluate_SIDD/evaluate_SIDD.py:63
 *   b200dn_ssim             skimage structural_similarity call sites evaluate_Unet_diffusion/evaluate_model.py:30-34,
 *                                                                    evaluate_SIDD/evaluate_SIDD.py:64
 *   b200dn_ssim_window      structural_similarity's other options (gaussian_weights, sigma, win_size,
 *                           use_sample_covariance, K1, K2, full): the SSIM of the published tables (Wang et al. 2004)
 *   b200dn_welch_psd        scipy.signal.welch(img.flatten(), nperseg=256)
 *                                                                    evaluate_Unet_diffusion/plot.py:155-157,233-235,287-290
 *   b200dn_patch_gather_image / b200dn_patch_gather / b200dn_maxpool3x3s2 / b200dn_lpips_head
 *                           lpips.LPIPS(net='alex') (lpips 0.1: ScalingLayer, AlexNet features[0:12] with the
 *                           convolutions on b200dn_igemm, the lin heads)      evaluate_Unet_diffusion/evaluate_model.py:46-71
 *   b200dn_l2pool3x3s2 / b200dn_dists_head
 *                           DISTS_pytorch.DISTS (DISTS 0.1: ImageNet normalisation through b200dn_patch_gather_image,
 *                           VGG16 features[0:30] on b200dn_igemm with L2pooling, the structure / texture head)
 *                                                                    evaluate_Unet_diffusion/evaluate_model.py:46-71
 *   b200dn_dihedral_expand / b200dn_dihedral_reduce
 *                           x8 geometric self-ensemble (the 8 flips / rotations of the image, each output
 *                           transformed back and averaged) around RDUNet.forward / improved_sampling
 *   b200dn_bm3d             bm3d.bm3d / bm3d.bm3d_rgb (the classical baseline, profile 'np' with a DCT in both
 *                           stages, colour in the opponent space)  evaluate_Unet_diffusion/evaluate_model.py
 *   b200dn_gauss_noise_u8   np.random.normal + clip + uint8 + ToTensor/Normalize
 *                                                                    dataset_creation/custom_dataset.py:83-87,
 *                                                                    dataset_creation/data_loader.py:35-38
 *   b200dn_u8_to_norm       ToTensor + Normalize(0.5, 0.5)           evaluate_SIDD/evaluate_SIDD.py:23-26,
 *                                                                    evaluate_SIDD/benchmark.py:35-36
 *   b200dn_norm_to_u8       (y+1)/2 -> clip(.*255) -> uint8          evaluate_SIDD/benchmark.py:42-44
 */
#ifndef B200DN_H_
#define B200DN_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200DN_ABI_VERSION 2

/* error codes */
#define B200DN_OK          0
#define B200DN_E_ARG      -1   /* bad argument (shape, alignment, enum)           */
#define B200DN_E_CUDA     -2   /* CUDA runtime / driver error, no sm_100 device   */
#define B200DN_E_UNSUP    -3   /* valid request the kernels do not support        */

/* storage / MMA precision of the 16-bit activation path */
#define B200DN_PREC_BF16     0  /* bf16 weights x bf16 activations, 1 MMA          */
#define B200DN_PREC_FP16     1  /* fp16 weights x fp16 activations, 1 MMA          */
#define B200DN_PREC_BF16X2   2  /* bf16 W x (bf16 hi + bf16 lo) activations, 2 MMA */
#define B200DN_PREC_BF16X3   3  /* (W hi+lo) x (A hi+lo) minus lo*lo, 3 MMA: fp32 validation build */
#define B200DN_PREC_FP16X2   4  /* fp16 W x (fp16 hi + fp16 lo) activations, 2 MMA              */

/* implicit-GEMM modes */
#define B200DN_MODE_CONV3X3  0  /* 3x3, stride 1, zero pad 1 (taps = 9)            */
#define B200DN_MODE_DOWN2X2  1  /* 2x2, stride 2 (taps = 4)                        */
#define B200DN_MODE_UP2X2    2  /* transposed 2x2, stride 2 (4 N-groups)           */
#define B200DN_MODE_CONV1X1  3  /* 1 tap, no shift (used by tests / microbenchmarks)*/

/* epilogue output kinds */
#define B200DN_OUT_NHWC16    0  /* 16-bit NHWC planes into a channel slice         */
#define B200DN_OUT_NCHW32    1  /* fp32 NCHW (+ fp32 NCHW residual), module boundary */

const char* b200dn_last_error(void);
int b200dn_abi_version(void);
/* number of SMs of the current device, or <0 */
int b200dn_sm_count(void);

/* ---- weight packing --------------------------------------------------------
 * Output layout (16-bit elements): [n_wplanes][groups][cout_pad][cin_pad], K(cin)-contiguous,
 * zero padded; cin_pad = roundup(Cin,64), cout_pad = roundup(Cout,16).
 * groups = kh*kw taps (conv) or 4 output phases ky*2+kx (convT).
 * n_wplanes = 2 only for B200DN_PREC_BF16X3 (hi, lo), else 1.
 * Conv2d weight is OIHW [Cout,Cin,kh,kw]; ConvTranspose2d weight is IOHW [Cin,Cout,2,2].
 */
int b200dn_pack_conv_weight(const float* w_oihw, int cout, int cin, int kh, int kw,
                            int prec, void* packed, void* stream);
int b200dn_pack_convt_weight(const float* w_iohw, int cin, int cout,
                             int prec, void* packed, void* stream);
/* bytes needed for a packed weight */
int64_t b200dn_packed_weight_bytes(int cout, int cin, int groups, int prec);

/* ---- the tensor-core implicit GEMM ---------------------------------------- */
typedef struct b200dn_igemm_args {
  int32_t mode;            /* B200DN_MODE_*                                          */
  int32_t prec;            /* B200DN_PREC_*                                          */
  int32_t B, H, W;         /* INPUT batch and spatial size (NHWC)                    */
  int32_t cin, cout;       /* logical channels (cout per phase for UP2X2)            */
  /* input activation planes: NHWC, `in_ctot` channels per pixel, the conv reads
     channels [0, cin).  in[1] is the "lo" plane (BF16X2/X3, FP16X2), else NULL.        */
  const void* in[2];
  int32_t in_ctot;
  const void* wpacked;     /* from b200dn_pack_*                                     */
  const float* bias;       /* [cout] fp32                                            */
  const float* slope;      /* [cout] fp32 PReLU slopes, NULL = no activation         */
  int32_t out_kind;        /* B200DN_OUT_*                                           */
  /* OUT_NHWC16: writes channels [out_coff, out_coff+cout) of out[] (out_ctot per pixel);
     output spatial size is HxW (CONV), H/2xW/2 (DOWN), 2Hx2W (UP).                  */
  void* out[2];
  int32_t out_ctot, out_coff;
  /* optional NHWC residual added after PReLU (dense-block `+ x`): channels [0,cout) */
  const void* res[2];
  int32_t res_ctot;
  /* OUT_NCHW32: out_nchw[B,cout,H,W] = prelu(conv) + res_nchw[b % res_bmod]        */
  float* out_nchw;
  const float* res_nchw;
  int32_t res_bmod;
  int32_t block_n;         /* 0 = auto; else UMMA N (multiple of 16, <= 256)         */
  int32_t max_ctas;        /* 0 = one per SM                                         */
  int32_t m_tiles;         /* 0 = auto; 1 or 2 A tiles (128 pixels each) per W tile  */
  int32_t impl;            /* CONV3X3 only: 0 = default, 1 = per-tap reload, 2 = haloed slab, 3 = haloed slab on CTA pairs */
  /* optional device int: OR'ed with 1 when an fp16-stored output value saturated at +-65504 (or was NaN).
     Ignored for bf16 storage (fp32 exponent range) and for OUT_NCHW32.  NULL = no watch.               */
  int32_t* sat_flag;
} b200dn_igemm_args;

int b200dn_igemm(const b200dn_igemm_args* args, void* stream);

/* Prepared launches.  b200dn_igemm validates, plans and encodes 2-3 CUtensorMaps on every call (~25 us of host time);
 * b200dn_igemm_prepare does that once and keeps the result, b200dn_igemm_launch / _launch_list only enqueue the
 * kernel(s) (one cudaLaunchKernelExC each).  A handle is bound to the pointers in `args` and to the device that was
 * current when it was prepared; only the OUT_NCHW32 output / residual pointers can be re-bound (they are the
 * caller's tensors at the module boundary and change from call to call).  Handles are not thread-safe objects:
 * do not rebind a handle while another thread launches it. */
typedef struct b200dn_igemm_prepared b200dn_igemm_prepared;
int b200dn_igemm_prepare(const b200dn_igemm_args* args, b200dn_igemm_prepared** out);
int b200dn_igemm_rebind_nchw(b200dn_igemm_prepared* prep, float* out_nchw, const float* res_nchw, int res_bmod);
int b200dn_igemm_launch(const b200dn_igemm_prepared* prep, void* stream);
int b200dn_igemm_launch_list(b200dn_igemm_prepared* const* preps, int n, void* stream);
void b200dn_igemm_release(b200dn_igemm_prepared* prep);

/* The launch configuration b200dn_igemm would choose for `args` on a device with `sm_count` SMs, without touching the
 * GPU (pointers are only checked for NULL).  Host-side tests sweep layer shapes through it to check that every choice
 * fits the kernels' shared-memory / TMEM budgets; tools print it next to measured times. */
typedef struct b200dn_igemm_plan_info {
  int32_t kernel;          /* 0 per-tap kernel, 1 slab kernel (one CTA per tile), 2 slab kernel on CTA pairs          */
  int32_t mt;              /* 128-pixel sub-tiles per CTA tile                                                        */
  int32_t block_n;         /* UMMA N                                                                                  */
  int32_t num_n_tiles;     /* N tiles (x4 phases for UP2X2)                                                           */
  int32_t num_tiles;       /* tiles (pair tiles for kernel 2)                                                         */
  int32_t grid;            /* CTAs launched                                                                           */
  int32_t wres;            /* weights resident in shared memory                                                       */
  int32_t num_slabs, slab_bytes;     /* slab ring (kernels 1, 2)                                                      */
  int32_t num_stages, stage_bytes;   /* W ring (kernels 1, 2) or A+W ring (kernel 0)                                  */
  int32_t w_taps;          /* filter taps per W ring stage                                                            */
  int32_t tmem_cols;       /* TMEM columns allocated (power of two, <= 512)                                           */
  int32_t epi_staged;      /* smem-transposed epilogue                                                                */
  int32_t data_bytes_used; /* bytes of rings (+ resident weights) this launch places in shared memory                 */
  int32_t data_bytes_budget; /* what the kernel's layout provides for them                                            */
} b200dn_igemm_plan_info;

int b200dn_igemm_plan(const b200dn_igemm_args* args, int sm_count, b200dn_igemm_plan_info* info);

/* ---- fused dense block --------------------------------------------------------
 * A whole DenoisingBlock (UNet/RDUNet_model.py:95-115: four chained 3x3 conv + PReLU over the growing concatenation,
 * then `+ x`) of the 32-channel level as ONE kernel: input-stationary passes whose partial sums stay in TMEM, o0..o2
 * only in shared memory.  Reads channels [0, 32) of `in`, writes channels [out_coff, out_coff + 32) of `out`
 * (NHWC 16-bit; `in` and `out` must be different buffers).  Same 16-bit rounding points as four b200dn_igemm launches.
 * Only channels == 32 and B200DN_PREC_BF16 / B200DN_PREC_FP16 are supported (B200DN_E_ARG otherwise).
 * The handle is launched / released with b200dn_igemm_launch[_list] / b200dn_igemm_release.                    */
typedef struct b200dn_dense_block_args {
  int32_t prec;
  int32_t B, H, W;
  int32_t channels;          /* C = 32; growth C / 2                                              */
  const void* in;            /* NHWC 16-bit, in_ctot channels per pixel                           */
  int32_t in_ctot;
  void* out;
  int32_t out_ctot, out_coff;
  const void* wfused;        /* from b200dn_pack_dense_block_weights                              */
  const float* bias[4];      /* conv_0..3 biases: 16, 16, 16, 32 floats                           */
  const float* slope[4];     /* actv_0..3 PReLU slopes, same shapes                               */
  int32_t max_ctas;          /* 0 = one per SM                                                    */
  int32_t* sat_flag;         /* optional fp16 saturation watch (see b200dn_igemm_args)            */
  int64_t* timeline;         /* optional diagnostics: CTA 0 writes up to 4096 (event, clock) pairs, entry 0 = count */
} b200dn_dense_block_args;
/* w0..w3: conv_0..3 weights, OIHW fp32 [16,32,3,3], [16,48,3,3], [16,64,3,3], [32,80,3,3]        */
int64_t b200dn_dense_block_weight_bytes(int channels);
int b200dn_pack_dense_block_weights(const float* w0, const float* w1, const float* w2, const float* w3,
                                    int channels, int prec, void* packed, void* stream);
int b200dn_dense_block_prepare(const b200dn_dense_block_args* args, b200dn_igemm_prepared** out);
/* Optional: hand the block's bias / PReLU slopes to a prepared dense block as HOST values (bias_host[j], slope_host[j]:
 * 16, 16, 16, 32 floats of conv_0..conv_3, the same numbers the device arrays of the args hold).  They then travel in
 * the launch parameters (constant bank) and the epilogue reads them as instruction operands instead of staging them in
 * shared memory — the kernel runs at the shared-memory bandwidth wall and the broadcast reads were 11 % of its
 * shared-memory wavefronts.  Results are bit-identical.  May be called again to refresh the values. */
int b200dn_dense_block_set_epilogue_constants(b200dn_igemm_prepared* prep, const float* const* bias_host,
                                              const float* const* slope_host);

/* ---- 2..4 DEPENDENT 3x3 convolutions of one resolution in one persistent launch (csrc/conv3x3_slab_sm100.cu) -------
 * layers[k] is a b200dn_igemm_args as b200dn_igemm takes it (MODE_CONV3X3, OUT_NHWC16, PREC_BF16 or PREC_FP16, all
 * tuning knobs 0, same B/H/W/prec).  Layer k may read anything written before the launch plus the outputs of layers
 * < k (the [x | o0 | o1 | o2] slices of a DenoisingBlock); no layer may write channels that it or an earlier layer of the
 * chain reads as input (checked).  A tile of layer k starts as soon as the 3 x 3 neighbourhood of tiles of layer k-1
 * is stored (per-tile counters in `workspace`), so the layers overlap and the pipelines never drain in between.
 * Results are bit-equal to launching the layers one by one.
 * workspace: device buffer of b200dn_conv_chain_workspace_bytes, 16-byte aligned, zero-filled ONCE by the caller and
 * owned by this handle afterwards (counters are monotonic across launches; no reset is needed).
 * Returns B200DN_E_UNSUP (handle NULL) when the layers do not all run on the CTA-pair kernel with one tiling, or
 * when a layer has fewer than two rounds of tiles per SM pair (batch 1-2: nothing to overlap, measured slower than
 * separate launches; flags = B200DN_CHAIN_FORCE builds the chain anyway) — launch them one by one then.
 * Launch with b200dn_igemm_launch / _launch_list.  Its CTAs wait on each other: chain launches on DIFFERENT streams
 * of one device must not overlap (env B200DN_CHAIN_COOP=1 makes the launch cooperative, which lifts this but cannot
 * run under ncu); one launch of a handle at a time. */
int64_t b200dn_conv_chain_workspace_bytes(const b200dn_igemm_args* layers, int n_layers);
#define B200DN_CHAIN_FORCE 1
int b200dn_conv_chain_prepare(const b200dn_igemm_args* layers, int n_layers, void* workspace, int flags,
                              b200dn_igemm_prepared** out);

/* ---- input block conv_1 (Cin = img_channels [+ 1]) ---------------------------------------------------------
 * Single-plane modes (BF16, FP16) with cout <= 256 run on tensor cores: 16-bit weights, the fp32 image (and t) gathered
 * as 16-bit hi + lo planes, fp32 accumulation.  Two-plane modes and cout > 256 run on CUDA cores in fp32.
 * x: fp32 NCHW [Bx,img_channels,H,W] (3 = RGB, 1 = grayscale); image b of the output reads x[b % Bx].
 * t: optional timestep plane source; element (b,y,x) = t[b*t_sb + y*t_sh + x*t_sw]
 *    (strides in elements, 0 = broadcast).  NULL -> no timestep channel.
 * w: OIHW fp32 [cout, img_channels (+1), 3, 3].  Output: NHWC 16-bit planes, channels [0,cout).
 * sat_flag: optional fp16 saturation watch, as in b200dn_igemm_args.
 */
int b200dn_conv_in(const float* x, int Bx, int img_channels, const float* t, int64_t t_sb, int64_t t_sh, int64_t t_sw,
                   int B, int H, int W, int cout,
                   const float* w, const float* bias, const float* slope,
                   int prec, void* out0, void* out1, int out_ctot, int32_t* sat_flag, void* stream);

/* ---- sampler elementwise ---------------------------------------------------- */
/* x_next = (x - ((1-a_t)*u1 + a_t*y)) + ((1-a_p)*u2 + a_p*y), fp32, reference op order.
   one_m_at etc. are the fp32-rounded python scalars.  n = element count.            */
int b200dn_sampler_step(const float* x, const float* u1, const float* u2, const float* y,
                        float one_m_at, float at, float one_m_ap, float ap,
                        float* x_next, int64_t n, void* stream);
/* out = alpha*noisy + (1-alpha)*clean */
int b200dn_lerp(const float* clean, const float* noisy, float alpha, float one_m_alpha,
                float* out, int64_t n, void* stream);

/* ---- metrics ------------------------------------------------------------------
 * Both reductions are two-pass and bit-reproducible: every block writes one partial sum into `workspace`
 * (device memory, 8-byte aligned, at least b200dn_*_workspace_bytes() bytes, contents undefined afterwards)
 * and a second kernel adds the partials of each image / plane in a fixed order.  No atomics.          */
int64_t b200dn_psnr_sse_workspace_bytes(int64_t n_images, int64_t n_per_image);
int64_t b200dn_ssim_workspace_bytes(int64_t n_planes, int H, int W);
/* sse[i] (fp64) = sum over the n_per_image elements of image i of (a-b)^2            */
int b200dn_psnr_sse(const float* a, const float* b, int64_t n_images, int64_t n_per_image,
                    double* sse, void* workspace, int64_t workspace_bytes, void* stream);
/* skimage-0.22-style SSIM (7x7 uniform window, sample covariance, crop 3, K1=.01 K2=.03)
   on fp32 planes: a,b are [n_planes,H,W]; ssim_sum[p] (fp64) = sum of S over the cropped
   interior of plane p (divide by (H-6)*(W-6) for the mean).  Window sums in fp32.     */
int b200dn_ssim(const float* a, const float* b, int64_t n_planes, int H, int W,
                float data_range, double* ssim_sum, void* workspace, int64_t workspace_bytes, void* stream);

/* skimage-0.22 SSIM with every option of structural_similarity: a separable filter of 2*radius+1 taps over scipy's
   'reflect' borders (d c b a | a b c d, repeated when the filter is wider than the plane), any covariance normaliser,
   C1 and C2, the crop (win_size-1)/2 and, optionally, the map of S over the whole plane.  Window sums in fp32.    */
#define B200DN_SSIM_MAX_RADIUS 15
typedef struct b200dn_ssim_window_opts {
  int32_t radius;          /* filter radius r, 0 .. B200DN_SSIM_MAX_RADIUS                                      */
  int32_t win_size;        /* odd, <= min(H, W): the crop is (win_size-1)/2 on every side                       */
  float cov_norm;          /* NP/(NP-1) with sample covariance (NP = win_size^2), else 1                        */
  float C1, C2;            /* (K1*R)^2, (K2*R)^2                                                                */
  /* weights[k], k = 0 .. 2r, multiplies the sample at offset k - r along each axis: gaussian_filter's taps, or
     1/win_size for uniform_filter (radius = (win_size-1)/2)                                                        */
  float weights[2 * B200DN_SSIM_MAX_RADIUS + 1];
} b200dn_ssim_window_opts;
int64_t b200dn_ssim_window_workspace_bytes(int64_t n_planes, int H, int W);
/* a,b: [n_planes,H,W] fp32.  ssim_sum[p] (fp64) = sum of S over the cropped interior of plane p (divide by
   (H-2*crop)*(W-2*crop) for the mean).  map: NULL, or [n_planes,H,W] fp32 that receives S at every pixel.
   A plane's results do not depend on n_planes.                                                                   */
int b200dn_ssim_window(const float* a, const float* b, int64_t n_planes, int H, int W,
                       const b200dn_ssim_window_opts* opts, double* ssim_sum, float* map,
                       void* workspace, int64_t workspace_bytes, void* stream);

/* Welch PSD with scipy.signal.welch's defaults at nperseg = 256 (fs = 1, periodic Hann, 50 % overlap, constant
   detrend, one-sided density scaling, mean over segments), float32 throughout like scipy for float32 input.
   x: [n_signals, n] fp32 (each row one flattened image, n >= 256); pxx: [n_signals, 129] fp32;
   frequencies are k/256, k = 0..128.  Two-pass, bit-reproducible (workspace as for the metrics above).  */
int64_t b200dn_welch_psd_workspace_bytes(int64_t n_signals, int64_t n);
int b200dn_welch_psd(const float* x, int64_t n_signals, int64_t n, float* pxx,
                     void* workspace, int64_t workspace_bytes, void* stream);

/* ---- LPIPS (lpips 0.1, net='alex') ----------------------------------------------
 * The trunk's convolutions are b200dn_igemm launches: conv1 (11x11/s4/p2) and conv2 (5x5/p2) as MODE_CONV1X1 GEMMs over
 * patch rows gathered here, conv3..conv5 as MODE_CONV3X3; ReLU is a PReLU with slopes 0.  Patch rows are NHWC 16-bit
 * planes [B, Ho, Wo, kpad] in (ky, kx, ci) order, zero padded to kpad columns (a multiple of 8 >= kh*kw*C); taps outside
 * the image are 0.  These entry points take the bf16-stored precisions only (BF16, BF16X2, BF16X3; B200DN_E_ARG else);
 * the lo planes are used for the two-plane ones. */
/* conv1 rows from the fp32 NCHW image pair: output image b < N reads in0[b], b >= N reads in1[b - N].  Each sample is
   x' = (x - shift[c]) / scale[c] in fp32 (x = 2x - 1 first when normalize != 0); padding is zeros of x'. */
int b200dn_patch_gather_image(const float* in0, const float* in1, int N, int C, int H, int W,
                              const float* shift, const float* scale, int normalize, int kh, int kw, int stride,
                              int pad, int kpad, int prec, void* out0, void* out1, void* stream);
/* rows from NHWC 16-bit planes [B, H, W, C] (C a multiple of 8) */
int b200dn_patch_gather(const void* in_hi, const void* in_lo, int B, int H, int W, int C, int kh, int kw,
                        int stride, int pad, int kpad, int prec, void* out0, void* out1, void* stream);
/* nn.MaxPool2d(3, 2) (floor mode, no padding) on NHWC 16-bit planes [B, H, W, C] -> [B, (H-3)/2+1, (W-3)/2+1, C].
   Two planes: the maximum of hi + lo wins and its (hi, lo) pair is copied. */
int b200dn_maxpool3x3s2(const void* in_hi, const void* in_lo, int B, int H, int W, int C, int prec,
                        void* out0, void* out1, void* stream);
/* One tap of the head: features NHWC [2N, H, W, C] (C a multiple of 8, <= 512; entries [0, N) are the in0 images,
   [N, 2N) their partners), lin weight [C] fp32. */
typedef struct b200dn_lpips_tap {
  const void* feat[2];     /* hi, lo planes (lo NULL for one-plane precisions)                            */
  const float* weight;
  int32_t H, W, C;
} b200dn_lpips_tap;
/* out[n] (fp32) = sum over taps l of mean over H_l x W_l of sum_c w_l[c] (f0/(|f0|+1e-10) - f1/(|f1|+1e-10))^2, the
   norms over channels, per pixel in fp32; spatial and tap sums in fp64.  Two-pass, bit-reproducible, and an image
   pair's value does not depend on N (workspace as for the metrics below). */
int64_t b200dn_lpips_head_workspace_bytes(const b200dn_lpips_tap* taps, int n_taps, int N);
int b200dn_lpips_head(const b200dn_lpips_tap* taps, int n_taps, int N, int prec, float* out,
                      void* workspace, int64_t workspace_bytes, void* stream);

/* ---- DISTS (DISTS_pytorch 0.1) --------------------------------------------------
 * The VGG16 convolutions are b200dn_igemm launches: conv1_1 as a MODE_CONV1X1 GEMM over the 3x3 patch rows of
 * b200dn_patch_gather_image (shift = ImageNet mean, scale = std, so the padding holds zeros of the normalised image),
 * the others MODE_CONV3X3; ReLU is a PReLU with slopes 0.  Same precisions as the LPIPS entry points above. */
/* DISTS' L2pooling: sqrt(conv2d(x^2, filter, stride 2, padding 1, groups C) + 1e-12) on NHWC 16-bit planes
   [B, H, W, C] -> [B, (H-1)/2+1, (W-1)/2+1, C]; filter fp32 [C][3][3] (the module's [C, 1, 3, 3] buffer).  fp32
   arithmetic on hi + lo, taps summed in (ky, kx) order. */
int b200dn_l2pool3x3s2(const void* in_hi, const void* in_lo, int B, int H, int W, int C, const float* filter, int prec,
                       void* out0, void* out1, void* stream);
/* One feature stage of the head: NHWC [2N, H, W, C] (C a multiple of 64; entries [0, N) are the in0 images, [N, 2N)
   their partners). */
typedef struct b200dn_dists_stage {
  const void* feat[2];     /* hi, lo planes (lo NULL for one-plane precisions)                            */
  int32_t H, W, C;
} b200dn_dists_stage;
/* out[n] (fp32) = 1 - sum_c (alpha[c] S1_c + beta[c] S2_c) / (sum alpha + sum beta) over the channels of stage 0 (the
   fp32 NCHW inputs in0 / in1 [N, 3, H, W] themselves) and then of stages[0..n_stages), alpha / beta fp32 [3 + sum C]
   in that order; S1 = (2 mx my + 1e-6) / (mx^2 + my^2 + 1e-6), S2 = (2 cov + 1e-6) / (vx + vy + 1e-6) with the
   population moments over H x W.  Moments and head in fp64.  Two-pass, bit-reproducible, an image pair's value does
   not depend on N, and swapping in0 / in1 (with the feature halves) gives the same bits. */
int64_t b200dn_dists_head_workspace_bytes(int H, int W, const b200dn_dists_stage* stages, int n_stages, int N);
int b200dn_dists_head(const float* in0, const float* in1, int H, int W, const b200dn_dists_stage* stages,
                      int n_stages, int N, const float* alpha, const float* beta, int prec, float* out,
                      void* workspace, int64_t workspace_bytes, void* stream);

/* ---- x8 geometric self-ensemble ------------------------------------------------
 * The transforms are the dihedral group of the square, k = 0..7, on fp32 NCHW planes (torch ops on [B, C, H, W]):
 *   T_k(x)    = torch.rot90(k < 4 ? x : torch.flip(x, [3]), k % 4, [2, 3])
 *   T_k^-1(y) = torch.rot90(y, -(k % 4), [2, 3]), then torch.flip(., [3]) if k >= 4
 * Even k keep H x W, odd k turn it into W x H, so the transformed batch is two groups of 4B images:
 *   group B200DN_DIHEDRAL_GROUP(k) (0 = even [4B, C, H, W], 1 = odd [4B, C, W, H]), image
 *   B200DN_DIHEDRAL_INDEX(k, b, B) of that group holds T_k(x[b]).
 * For square images the odd group may directly follow the even one in memory: one [8B, C, H, W] batch.  Any H, W,
 * C, B >= 1; `x`, `even`, `odd` and `out` must not overlap. */
#define B200DN_DIHEDRAL_GROUP(k) ((k) & 1)
#define B200DN_DIHEDRAL_INDEX(k, b, B) (((k) >> 1) * (B) + (b))
/* even[...] = T_k(x) for the even k, odd[...] = T_k(x) for the odd k: one read, eight writes */
int b200dn_dihedral_expand(const float* x, int B, int C, int H, int W, float* even, float* odd, void* stream);
/* out[B, C, H, W] = (((y_0 + y_1) + y_2) + ... + y_7) * 0.125 in fp32, adds in k order, y_k = T_k^-1 of the images
   of `even` / `odd` that hold transform k (layout as above) */
int b200dn_dihedral_reduce(const float* even, const float* odd, int B, int C, int H, int W, float* out, void* stream);

/* ---- BM3D / CBM3D --------------------------------------------------------------
 * Dabov et al. 2007, both stages, on fp32 [B, C, H, W] images in [0, 1] (C = 1 grey, C = 3 RGB through the opponent
 * space; all channels share the groups matched on its first channel).  8 x 8 blocks; reference blocks at rows
 * {0, 3, 6, ...} u {H - 8}, columns alike; candidates within +-19 rows / columns (clipped at the border); matching on
 * q = rint(1024 * Y) with d = sum (q_R - q)^2 kept iff d <= floor(tau * 64 * 2^20 / 255^2) (tau 3000 / 400); the group
 * is the reference then the kept candidates in ascending (d, r, c), cut to N2 (16 / 32), then to a power of two.
 * 2-D orthonormal DCT + Haar along the group; stage 1 hard-thresholds at 2.7 sigma_c, stage 2 is the Wiener filter on
 * the basic estimate; Kaiser (beta 2) weighted aggregation with 64-bit fixed-point sums, so the output is
 * bit-reproducible and an image's result does not depend on its batch.
 *   sigma : [B] fp32 on the device, noise standard deviation in the image's units
 *   basic : optional [B, C, H, W] fp32 basic estimate; when given, only stage 2 runs (stages must be 3)
 *   stages: B200DN_BM3D_HARD_THRESHOLDING (stage 1 only) or B200DN_BM3D_ALL_STAGES
 *   match1 / size1, match2 / size2: optional group outputs of stage 1 / 2: [B, NREF(H), NREF(W), N2] int32 positions
 *           r * W + c in group order padded with -1 (N2 = B200DN_BM3D_N2_HT / _WIE), [B, NREF(H), NREF(W)] int32 sizes
 * H, W >= 8, H * W < 2^31.  out must not overlap the inputs.  The workspace holds fp64 planes and 64-bit sums:
 * b200dn_bm3d_workspace_bytes(args) bytes (about 40 B per pixel and channel). */
#define B200DN_BM3D_HARD_THRESHOLDING 1
#define B200DN_BM3D_ALL_STAGES 3
#define B200DN_BM3D_N2_HT 16
#define B200DN_BM3D_N2_WIE 32
#define B200DN_BM3D_NREF(n) (((n) - 8) / 3 + 1 + (((n) - 8) % 3 != 0))
typedef struct b200dn_bm3d_args {
  const float* z;          /* [B, C, H, W] noisy images */
  const float* basic;      /* optional [B, C, H, W] basic estimate (stage 2 only) */
  const float* sigma;      /* [B] device */
  int B, C, H, W;
  int stages;
  float* out;              /* [B, C, H, W] */
  int32_t* match1;         /* optional [B, NREF(H), NREF(W), 16] */
  int32_t* size1;          /* optional [B, NREF(H), NREF(W)] */
  int32_t* match2;         /* optional [B, NREF(H), NREF(W), 32] */
  int32_t* size2;          /* optional [B, NREF(H), NREF(W)] */
} b200dn_bm3d_args;
int64_t b200dn_bm3d_workspace_bytes(const b200dn_bm3d_args* args);
int b200dn_bm3d(const b200dn_bm3d_args* args, void* workspace, int64_t workspace_bytes, void* stream);

/* ---- noise synthesis / data formats ------------------------------------------- */
/* clean_u8: [B,H,W,C] uint8 (HWC as in PIL / the SIDD .mat blocks).
   noisy_u8 (optional, same layout), noisy_norm (optional) fp32 NCHW in [-1,1],
   clean_norm (optional) fp32 NCHW.  sigma[b] per image.  Philox4x32-10,
   key=(seed_lo,seed_hi), counter=(elem_idx/4 lo, hi, stream_id, 0), Box-Muller.     */
int b200dn_gauss_noise_u8(const uint8_t* clean_u8, int B, int H, int W, int C,
                          const float* sigma, uint64_t seed, uint32_t stream_id,
                          uint8_t* noisy_u8, float* noisy_norm, float* clean_norm, void* stream);
/* raw fp32 standard normals z[i], same generator (for pinning the RNG itself)        */
int b200dn_philox_normal(float* z, int64_t n, uint64_t seed, uint32_t stream_id, void* stream);
/* u8 HWC [B,H,W,C] -> fp32 NCHW (x/255 - 0.5)/0.5 */
int b200dn_u8_to_norm(const uint8_t* in, int B, int H, int W, int C, float* out, void* stream);
/* fp32 NCHW in [-1,1] -> u8 HWC: trunc(clip((y+1)/2*255, 0, 255)) */
int b200dn_norm_to_u8(const float* in, int B, int H, int W, int C, uint8_t* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* B200DN_H_ */
