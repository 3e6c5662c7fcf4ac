/*
 * libdvc.so -- C ABI of the B200-native exemplar-video-colorization forward path.
 *
 * The reference (zhangmozhe/Deep-Exemplar-based-Video-Colorization) has no FFI of its own: its
 * hot path is three Python nn.Module.forward() methods plus per-frame glue.  Each entry point below
 * names the reference interface it replaces (file:line relative to the reference root).  The
 * Python drop-in modules (models/NonlocalNet.py, models/ColorVidNet.py in the package) bind these
 * symbols with ctypes; INTEGRATION.md shows that binding.
 *
 * Conventions
 *   - plain pointers and sizes only; no torch / C++ types cross the boundary.
 *   - tensors are fp32, contiguous, NCHW unless stated; `dev_*` pointers are device memory on the
 *     context's device, `host_*` pointers are host memory (pinned for the async paths).
 *   - every function returns DVC_OK (0) or a negative dvc_status; dvc_last_error() gives the text.
 *   - all device work is enqueued on the `stream` argument (a cudaStream_t passed as void*); no
 *     entry point synchronises the device unless stated.
 *   - there is NO CPU fallback: without a CUDA device every compute entry point fails with
 *     DVC_ERR_CUDA.
 *   - legal frame shapes are the reference's (SURVEY.md fact 2): H % 8 == 0, W % 16 == 0, H,W >= 16;
 *     anything else returns DVC_ERR_SHAPE (the reference raises RuntimeError at NonlocalNet.py:464).
 */
#ifndef DVC_H_
#define DVC_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct dvc_ctx dvc_ctx;

typedef enum dvc_status {
  DVC_OK = 0,
  DVC_ERR_ARG = -1,     /* null pointer, unknown key, unsupported option (pool="avg", WTA_scale_weight != 1) */
  DVC_ERR_SHAPE = -2,   /* illegal H/W or mismatching tensor shape */
  DVC_ERR_CUDA = -3,    /* CUDA runtime error (text in dvc_last_error) or no device */
  DVC_ERR_STATE = -4,   /* weights missing, exemplar not set, ... */
  DVC_ERR_NCCL = -5
} dvc_status;

typedef enum dvc_net { DVC_NET_VGG = 0, DVC_NET_WARP = 1, DVC_NET_COLOR = 2 } dvc_net;

/* Arithmetic used by the GEMM-shaped kernels (convolutions, correlation).
 *   DVC_MATH_FP32    CUDA-core fp32 FMA (exact fp32 products, two-level accumulation; the on-GPU fp32 reference)
 *   DVC_MATH_TF32X3  tcgen05 kind::tf32 on hi/lo split operands, 3 MMAs per product, TMEM chunk sums promoted
 *                    to fp32 registers (fp32-class accuracy; THE DEFAULT for convolutions and correlation)
 *   DVC_MATH_BF16X3  tcgen05 kind::f16 (bf16) on hi/lo split operands (correlation only; fast mode, |df| ~ 2e-6)
 *   DVC_MATH_FP16X3  tcgen05 kind::f16 (fp16) on hi/lo planes of x * 2^14 (correlation only: its operands are unit
 *                    vectors, so the power-of-two scale is exact): tf32x3's 2 x 11 bits at bf16x3's speed
 */
typedef enum dvc_math { DVC_MATH_FP32 = 0, DVC_MATH_TF32X3 = 1, DVC_MATH_BF16X3 = 2, DVC_MATH_FP16X3 = 3 } dvc_math;

/* ---- lifetime ------------------------------------------------------------------------------- */

/* One context per device (reference: test.py:147-166 builds one set of modules on cuda:0).
 * Not thread-safe per context. */
int dvc_create(dvc_ctx** out, int device);
int dvc_destroy(dvc_ctx* ctx);
const char* dvc_last_error(const dvc_ctx* ctx); /* ctx may be NULL: last create() error */
const char* dvc_version(void);

/* Select the arithmetic of the conv layers and of the correlation (see dvc_math). */
int dvc_set_math(dvc_ctx* ctx, int conv_math, int corr_math);

/* ---- weights: replaces nn.Module.load_state_dict (test.py:150,158-159) ----------------------- */

/* `data` holds the tensor for `key` exactly as in the reference state_dict (OIHW fp32 for conv
 * weights, [C] for biases, [1] for PReLU slopes, [C,1,1,1] for the depthwise *_ss scales).
 * `data` may be a host or a device pointer (cudaMemcpyDefault).  Synchronous. */
int dvc_set_weight(dvc_ctx* ctx, int net, const char* key, const float* data, const int64_t* shape, int ndim);

/* ---- module-level drop-ins ------------------------------------------------------------------ */

/* VGG19_pytorch.forward(x, out_keys, preprocess) -- models/NonlocalNet.py:228-256.
 * dev_x [B,3,H,W] RGB in [0,1].  keys[i] in {"r11".."r54","p1".."p5"}; dev_out[i] receives that map
 * (NCHW fp32, caller-allocated).  Like the reference, preprocess != 0 applies util.py:347-352. */
int dvc_vgg19_forward(dvc_ctx* ctx, const float* dev_x, int B, int H, int W, int preprocess,
                      const char* const* keys, float* const* dev_out, int n_keys, void* stream);

/* WarpNet.forward(B_lab_map, A_relu2_1..5_1, B_relu2_1..5_1, temperature, ...) --
 * models/NonlocalNet.py:427-502.  dev_A[4]/dev_Bf[4] are the (already feature_normalize()d) r22,r32,r42,r52
 * maps: [B,128,H/2,W/2], [B,256,H/4,W/4], [B,512,H/8,W/8], [B,512,H/16,W/16].
 * dev_y [B,3,H,W], dev_sim [B,1,H,W].  reuse_exemplar != 0 skips the B-side recomputation and uses the
 * phi / pooled-Lab operands cached by the previous call (valid only for identical B tensors).
 * wta_scale_weight must be 1 (the reference bypasses WTA_scale in that case, NonlocalNet.py:486). */
int dvc_warpnet_forward(dvc_ctx* ctx, const float* dev_B_lab_map, const float* const* dev_A,
                        const float* const* dev_Bf, int B, int H, int W, float temperature,
                        float wta_scale_weight, int reuse_exemplar, float* dev_y, float* dev_sim, void* stream);

/* ColorVidNet.forward(x) -- models/ColorVidNet.py:96-144.  dev_x [B,7,H,W] -> dev_out [B,2,H,W]. */
int dvc_colorvidnet_forward(dvc_ctx* ctx, const float* dev_x, int B, int H, int W, float* dev_out, void* stream);

/* ---- the correlation kernel on its own (microbench / unit-test entry) ------------------------ */

/* f = theta_hat^T phi_hat; sim = rowmax f; P = softmax_j(f/T); y = P V   (NonlocalNet.py:477-498)
 * dev_theta_hat [B,C,NA], dev_phi_hat [Bphi,C,NB] (Bphi == B or 1: one exemplar shared by B frames),
 * dev_V [Bphi,NB,3]; outputs dev_y [B,NA,3], dev_sim [B,NA]; dev_argmax [B,NA] int32 may be NULL.
 * C must be a multiple of 64 (256 = WarpNet.inter_channels, NonlocalNet.py:360; other depths, e.g. the patch features of
 * NonlocalWeightedAverage, NonlocalNet.py:95-108, take the exact 3-pass kernel). */
int dvc_corr_softmax_warp(dvc_ctx* ctx, const float* dev_theta_hat, const float* dev_phi_hat,
                          const float* dev_V, int B, int Bphi, int NA, int NB, int C, float temperature,
                          float* dev_y, float* dev_sim, int32_t* dev_argmax, void* stream);

/* ---- fused per-frame / per-clip path (test.py:57-96 + FrameColor.py:41-67) -------------------- */

/* Exemplar prologue, test.py:57-66: IB_lab [1,3,H,W] (centred L, a, b) -> sRGB -> VGG -> heads ->
 * phi_hat / pooled Lab, cached in the context.  Host or device pointer. */
int dvc_set_exemplar(dvc_ctx* ctx, const float* IB_lab, int H, int W, void* stream);

/* frame_colorization (FrameColor.py:41-67) for B frames against the cached exemplar.
 * IA_l [B,1,H,W] centred luminance; IA_last_lab [B,3,H,W]; out_ab [B,2,H,W];
 * optional out_warp_lab [B,3,H,W] and out_sim [B,1,H,W] (may be NULL).  All device pointers. */
int dvc_colorize_frames(dvc_ctx* ctx, const float* dev_IA_l, const float* dev_IA_last_lab, int B, int H, int W,
                        float temperature, float* dev_out_ab, float* dev_out_warp_lab, float* dev_out_sim,
                        void* stream);

/* A whole segment with the frame-to-frame recurrence of test.py:76-96 kept on the device:
 * host_L [F,1,H,W] (pinned) is copied in frame by frame, frame t's predicted ab feeds frame t+1,
 * host_ab [F,2,H,W] (pinned) receives the predictions.  first_last_lab: NULL = zeros (test.py:80) or a
 * host [1,3,H,W] tensor (test.py:78, --frame_propagate).  Synchronises `stream` before returning. */
int dvc_colorize_clip(dvc_ctx* ctx, const float* host_L, int F, int H, int W, float temperature,
                      const float* host_first_last_lab, float* host_ab, void* stream);

/* ---- pre / post-processing around the nets (SURVEY.md §8f row 1) ------------------------------ */

/* F.interpolate(x, scale_factor=0.5, mode="bilinear") -- test.py:58,71.  dev_src [planes,H,W] (H, W even) ->
 * dev_dst [planes,H/2,W/2]; planes = B*C of a contiguous NCHW tensor. */
int dvc_resize_half(dvc_ctx* ctx, const float* dev_src, int planes, int H, int W, float* dev_dst, void* stream);
/* F.interpolate(x, scale_factor=2, mode="bilinear") * scale -- test.py:100-102 (scale = 1.25 there).
 * dev_src [planes,h,w] -> dev_dst [planes,2h,2w]. */
int dvc_upsample2_scaled(dvc_ctx* ctx, const float* dev_src, int planes, int h, int w, float scale, float* dev_dst,
                         void* stream);

/* Output colour conversion of test.py:116-119 = utils/util.py:134-151 (batch_lab2rgb_transpose_mc for one image):
 * Lab = (l + 50, ab) -> skimage.color.lab2rgb (float64: D65 / 2-degree white point, z < 0 -> 0, the 0.2068966 cube
 * threshold, rgb_from_xyz = inv(xyz_from_rgb), sRGB gamma) -> clip [0,1] -> * 255 -> truncation to uint8.
 * dev_l [B,1,H,W] (centred L), dev_ab [B,2,H,W] -> dev_rgb [B,H,W,3] uint8 (the layout cv2 / PIL write). */
int dvc_lab_to_rgb8(dvc_ctx* ctx, const float* dev_l, const float* dev_ab, int B, int H, int W, unsigned char* dev_rgb,
                    void* stream);

/* Ingest colour conversion of test.py:44-45 = RGB2Lab + ToTensor + Normalize (utils/util_distortion.py:18-23,85-100):
 * skimage.color.rgb2lab in float64 (uint8 / 255, inverse sRGB gamma, xyz_from_rgb, D65 / 2-degree white point,
 * 0.008856 cube-root threshold), cast to float32, then L - 50.  dev_rgb [B,H,W,3] uint8 -> dev_lab [B,3,H,W]. */
int dvc_rgb8_to_lab(dvc_ctx* ctx, const unsigned char* dev_rgb, int B, int H, int W, float* dev_lab, void* stream);

/* ContextualLoss_forward.forward(X_features, Y_features, h, feature_centering) (models/ContextualLoss.py:82-126; the default
 * "forward" matching direction of train.py:79), VALUE ONLY -- no backward pass, so it serves evaluation, not training.
 * dev_X [B,C,NX], dev_Y [B,C,NY] (the reference's [B,C,h,w] feature maps, positions flattened), C a multiple of 64;
 * dev_loss [B] = -log(mean_i max_j A_ij).  Runs K7 twice: row maxima, then the online softmax with the per-row temperature
 * h * (1 - max_j f_ij + 1e-5).  Needs a tensor-core correlation mode. */
int dvc_contextual_loss_forward(dvc_ctx* ctx, const float* dev_X, const float* dev_Y, int B, int C, int NX, int NY, float h,
                                int feature_centering, float* dev_loss, void* stream);

/* The "WLS filter" of test.py:105-112: cv2.ximgproc.createFastGlobalSmootherFilter(guide, lambda, sigma_color,
 * lambda_attenuation = 0.25, num_iter = 3).filter(plane) for `planes` fp32 planes [planes,H,W] sharing one single-channel uint8
 * guide [H,W] (Min et al., Fast Global Image Smoothing Based on Weighted Least Squares, TIP 2014: per iteration a horizontal
 * and a vertical sweep of tridiagonal solves (I + lambda_n L) u = f, weights exp(-|dg| / sigma_color), lambda_{n+1} =
 * lambda_n * lambda_attenuation).  dev_dst may equal dev_src.  test.py uses lambda = 500, sigma_color = 4. */
int dvc_fgs_filter(dvc_ctx* ctx, const unsigned char* dev_guide, const float* dev_src, int planes, int H, int W, float lambda,
                   float sigma_color, float lambda_attenuation, int num_iter, float* dev_dst, void* stream);
/* The guide of test.py:106: uint8(uncenter_l(L) * 255 / 100) from the centred luminance plane dev_l [H,W]. */
int dvc_l_to_guide8(dvc_ctx* ctx, const float* dev_l, int H, int W, unsigned char* dev_guide, void* stream);

/* The resize inside CenterPad (utils/util_distortion.py:217-258) and the crop / pad around it:
 * skimage.transform.resize(I, (Hr, Wr), mode="reflect", preserve_range=True, clip=False, anti_aliasing=True) of the uint8
 * image dev_src [Hs,Ws,3] -- float64 Gaussian pre-filter with sigma = max(0, (in/out - 1)/2) per axis (scipy.ndimage
 * gaussian_filter, mode "mirror", truncate 4) then bilinear scipy.ndimage.zoom(order=1, mode="mirror", grid_mode=True) --
 * truncated to uint8; dev_dst [Ho,Wo,3] receives resized[y + oy, x + ox] where that exists and 0 elsewhere (CenterPad's
 * centred crop and torchvision CenterCrop's zero pad; the geometry is computed by the caller, dvc/prepost.py). */
int dvc_resize_antialias_crop_rgb8(dvc_ctx* ctx, const unsigned char* dev_src, int Hs, int Ws, int Hr, int Wr, int oy, int ox,
                                   unsigned char* dev_dst, int Ho, int Wo, void* stream);

/* ---- whole frames in, whole frames out ------------------------------------------------------------- */

/* Frame ingest of test.py:44-46,71 for F frames dev_src [F,Hs,Ws,3] (uint8 sRGB, same size): CenterPad resize + crop / pad
 * to [Ho,Wo] (geometry as for dvc_resize_antialias_crop_rgb8), sRGB -> Lab, and only the centred L is kept:
 * dev_l [F,1,Ho,Wo] at full size and dev_l_half [F,1,Ho/2,Wo/2] (dvc_resize_half of it).  Bit for bit the chain
 * dvc_resize_antialias_crop_rgb8 -> dvc_rgb8_to_lab -> channel 0 -> dvc_resize_half.  Ho and Wo must be even. */
int dvc_ingest_rgb8(dvc_ctx* ctx, const unsigned char* dev_src, int F, int Hs, int Ws, int Hr, int Wr, int oy, int ox, int Ho,
                    int Wo, float* dev_l, float* dev_l_half, void* stream);
/* Output side of test.py:99-119 for F frames: ab at half size dev_ab_half [F,2,Ho/2,Wo/2] -> x2 * 1.25 -> (wls != 0) the
 * Fast Global Smoother of each frame's two planes guided by its own luminance dev_l [F,1,Ho,Wo] (lambda, sigma_color,
 * attenuation 0.25, 3 iterations) -> sRGB uint8 dev_rgb [F,Ho,Wo,3].  Bit for bit dvc_upsample2_scaled(1.25) -> per frame
 * dvc_l_to_guide8 + dvc_fgs_filter -> dvc_lab_to_rgb8, in one launch per step for all F frames. */
int dvc_postprocess_rgb8(dvc_ctx* ctx, const float* dev_l, const float* dev_ab_half, int F, int Ho, int Wo, int wls, float lambda,
                         float sigma_color, unsigned char* dev_rgb, void* stream);
/* Colourise K consecutive frames of a clip, uint8 sRGB in and out: host_src [K,Hs,Ws,3] -> dvc_ingest_rgb8 -> the networks
 * with the recurrence of test.py:76-96 (as dvc_colorize_clip) -> dvc_postprocess_rgb8 -> host_dst [K,Ho,Wo,3].  The nets
 * run at Ho/2 x Wo/2, which must be the size of the exemplar given to dvc_set_exemplar.  continue_clip = 0 starts the
 * recurrence from zeros (test.py:80); continue_clip = 1 continues it from the last frame of the previous call, which
 * must have succeeded against the same exemplar and the same Ho x Wo (otherwise DVC_ERR_STATE) -- the source size may
 * change between calls.  A clip of any length can so be fed in chunks: device memory depends on the frame sizes only,
 * never on K.  host_src / host_dst may be host (pinned for full overlap) or device memory.  Synchronises `stream`
 * before returning. */
int dvc_colorize_video_rgb8(dvc_ctx* ctx, const unsigned char* host_src, int K, int Hs, int Ws, int Hr, int Wr, int oy, int ox,
                            int Ho, int Wo, float temperature, int wls, float lambda, float sigma_color, int continue_clip,
                            unsigned char* host_dst, void* stream);

/* ---- multi-GPU: exemplar operands travel once per clip (SURVEY.md §8e) ----------------------- */

/* ---- single-frame scaling: query-row-sharded correlation with a fused all-gather (SURVEY.md §8e, BASELINE config 4) --
 * Every row of NonlocalNet.py:477-498 is independent, so G GPUs can each take N/G query rows of one frame against the
 * full exemplar side.  Instead of an NCCL all-gather after the kernel, the kernel that finalises a result row stores it
 * into the full-size result buffer of EVERY GPU through peer-mapped pointers (NVLink stores).  The buffers are plain
 * cudaMalloc allocations shared between the one-process-per-GPU ranks with CUDA IPC. */

/* Allocate `bytes` of device memory and return its IPC handle (64 bytes, cudaIpcMemHandle_t) for the other ranks. */
int dvc_peer_buffer_create(dvc_ctx* ctx, int64_t bytes, void** dev_ptr, unsigned char* handle64);
/* Map another rank's buffer (handle from its dvc_peer_buffer_create) into this process; enables peer access. */
int dvc_peer_buffer_open(dvc_ctx* ctx, const unsigned char* handle64, void** dev_ptr);
int dvc_peer_buffer_close(dvc_ctx* ctx, void* opened_ptr);
int dvc_peer_buffer_destroy(dvc_ctx* ctx, void* created_ptr);
/* Until cleared with n = 0, dvc_corr_softmax_warp (B = 1) additionally stores row r of its result as global row
 * row0 + r into y4[g] ([N_total][4] floats: L, a, b, 0) and sim[g] ([N_total]) for g < n <= 8. */
int dvc_corr_set_peer_outputs(dvc_ctx* ctx, int n, float* const* y4, float* const* sim, int64_t row0);

/* Size in floats of the packed exemplar operands (phi_hat planes + pooled Lab) for an HxW exemplar. */
int64_t dvc_exemplar_pack_size(const dvc_ctx* ctx, int H, int W);
/* Pack the cached exemplar operands into / install them from a flat device buffer, so that the
 * caller can move them with ncclBroadcast (torch.distributed.broadcast) over NVLink. */
int dvc_exemplar_export(dvc_ctx* ctx, float* dev_buf, int64_t n_floats, void* stream);
int dvc_exemplar_import(dvc_ctx* ctx, const float* dev_buf, int64_t n_floats, int H, int W, void* stream);

/* ---- introspection -------------------------------------------------------------------------- */

/* Number of kernels this library launched since the last call with reset != 0. */
int64_t dvc_launch_count(dvc_ctx* ctx, int reset);
/* CUDA-event timing of the correlation kernel: mean milliseconds over the launches recorded since
 * the last reset (0 if none).  Recording is enabled with dvc_profile_corr(ctx, 1). */
int dvc_profile_corr(dvc_ctx* ctx, int enable);
double dvc_corr_mean_ms(dvc_ctx* ctx, int reset);
/* Same for the tensor-core convolution launches: dvc_conv_profile sums the CUDA-event durations (ms) and the
 * algorithmic FLOPs of the recorded launches of one kernel variant (64 / 128 / 256 = pixel-major channel tile,
 * 1 = channel-major kernel, 0 = all) and returns the number of launches. */
int dvc_profile_conv(dvc_ctx* ctx, int enable);
int dvc_conv_profile(dvc_ctx* ctx, int variant, int reset, double* total_ms, double* total_flops);

/* Debug / test hooks (not part of the drop-in surface).
 *   dvc_debug_set_flag: "two_level" (default 1) selects per-tap two-level fp32 accumulation in the
 *   CUDA-core convolution (shorter rounding chain; 0 = plain sequential accumulation, faster).
 *   dvc_debug_get_buffer: device pointer / size of a named internal workspace (padded NHWC activations
 *   carry their [B,H,W,C,P] signature in sig5) so tests can check intermediate stages. */
int dvc_debug_set_flag(dvc_ctx* ctx, const char* name, int value);
int dvc_debug_get_buffer(dvc_ctx* ctx, const char* name, void** dev_ptr, int64_t* bytes, int* sig5);
/*   dvc_debug_conv2d: ONE convolution layer (the weights `name` of network `net`, already set with dvc_set_weight) on a
 *   device NCHW input, through exactly the engine / operand format / epilogue the layer programs would use under the
 *   current dvc_set_math and debug flags ("tc_force_bn" = 64 / 128 / 256 pins the channel tile) -- the per-layer parity
 *   tests compare it with an fp64 F.conv2d (nn.Conv2d at NonlocalNet.py:235-255,364-423, ColorVidNet.py:96-143).
 *   pad_mode 0 = zero padding, 1 = ReflectionPad2d; act 0 none / 1 ReLU / 2 LeakyReLU(slope); in_bound >= max |x|
 *   (fixes the exact power-of-two scale of the fp16 operand planes); out_planes = 1 stores the result as fp16 hi/lo
 *   planes with the device-derived exponent and reads it back; upconv = 1: Upsample(2, nearest) + Conv2d(3x3) as four
 *   phase convolutions (y is [B][Cout][2H][2W]); fuse_tail = 1: conv10_2 + LeakyReLU + conv10_ab + tanh*128 (y is
 *   [B][2][H][W]); add: optional device NCHW addend of the output's shape; stats_out: optional device [B][Cout][2]
 *   doubles receiving (sum, sum of squares) over positions. */
int dvc_debug_conv2d(dvc_ctx* ctx, int net, const char* name, const float* dev_x, int B, int H, int W, int dil, int stride,
                     int act, float slope, int pad_mode, int upconv, int fuse_tail, float in_bound, int out_planes,
                     const float* dev_add, float* dev_y, double* dev_stats_out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DVC_H_ */
