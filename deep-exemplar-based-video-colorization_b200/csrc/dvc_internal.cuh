// Internal declarations shared by the kernels and the host-side layer programs of libdvc.so.
//
// Data layout in HBM (DESIGN.md §3): every activation is a "padded NHWC" fp32 tensor
//     [B][H + 2P][W + 2P][C]
// whose border of width P already holds what the consumer's padding mode would produce (zeros for
// the VGG / ColorVidNet convolutions, mirrored pixels for WarpNet's ReflectionPad2d).  With that
// layout a 3x3 (dilated) convolution is a plain GEMM over the flat padded pixel index p:
//     Y[p, co] = sum_tap sum_ci X[p + off(tap), ci] * Wt[tap][ci][co],  off = (dy*Wp + dx)*dil
// i.e. nine row-shifted [pixels x Cin] operands that TMA (or float4 loads) can fetch as ordinary
// 2-D tiles.  Border pixels compute garbage that the epilogue masks out.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace dvc {

// Device-side scale record of an fp16-plane activation whose range is only known at run time (conv -> ReLU -> conv
// chains).  The producer derives a rigorous bound of its outputs from the measured max |input| and the L1 norm of its
// weights, stores planes of value * 2^e, and leaves the measured max |output| for the next layer.
struct ScaleCell {
  unsigned int amax_bits;  // float bits of max |value| (non-negative floats order like unsigned ints), atomicMax
  int e;                   // exponent the planes were written with
};

struct DynOut {
  void* h16 = nullptr;                 // fp16 hi / lo output planes (same geometry as the fp32 destination) or nullptr
  void* l16 = nullptr;
  ScaleCell* cell_out = nullptr;       // max |output| (always, when set) and the exponent used (when h16 is set)
  const ScaleCell* cell_in = nullptr;  // dynamic input: exponent of its planes and its max |value| ...
  float in_bound = 0.f;                // ... or a static bound of |input|
  const ScaleCell* cell_add = nullptr;
  float add_bound = 0.f;
  float w_l1 = 0.f, b_max = 0.f, gain = 1.f;  // max_o sum |w[o]|, max |bias|, max(1, |activation slope|)
};

#ifdef __CUDACC__
__device__ __forceinline__ float exp2_int(int e) { return __int_as_float((127 + e) << 23); }  // e in [-126, 127]
// largest e with bound * 2^e <= 2^15 (fp16 max is 65504: one binade of slack), clamped
__device__ __forceinline__ int e16_from_bound(float bound) {
  if (!(bound > 0.f)) return 24;
  if (!(bound < 3.0e38f)) return -100;
  int ex;
  (void)frexpf(bound, &ex);  // bound = m * 2^ex, m in [0.5, 1)  ->  bound <= 2^ex
  const int e = 15 - ex;
  return e > 24 ? 24 : (e < -100 ? -100 : e);
}
__device__ __forceinline__ int dyn_out_exponent(const DynOut& d) {
  const float ain = d.cell_in ? __uint_as_float(d.cell_in->amax_bits) : d.in_bound;
  const float aadd = d.cell_add ? __uint_as_float(d.cell_add->amax_bits) : d.add_bound;
  const float bound = (fmaf(ain, d.w_l1, d.b_max) + aadd) * d.gain * 1.0001f;
  return e16_from_bound(bound);
}
__device__ __forceinline__ void warp_amax_commit(float amax, ScaleCell* cell) {
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, off));
  if ((threadIdx.x & 31) == 0 && amax > 0.f) atomicMax(&cell->amax_bits, __float_as_uint(amax));
}
// block-wide variant (blockDim.x <= 1024, every thread calls it): one atomic per block; `red` holds >= 32 floats
// (or as many as the block has warps)
__device__ __forceinline__ void block_amax_commit(float amax, ScaleCell* cell, float* red) {
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, off));
  const int w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  if ((threadIdx.x & 31) == 0) red[w] = amax;
  __syncthreads();
  if (threadIdx.x == 0) {
    float m = red[0];
    for (int i = 1; i < nw; ++i) m = fmaxf(m, red[i]);
    if (m > 0.f) atomicMax(&cell->amax_bits, __float_as_uint(m));
  }
}
// util_distortion.py:18-23 -> skimage.color.rgb2lab of one sRGB uint8 pixel in float64, then ToTensor (.float()) and
// Normalize (L - 50).  Shared by rgb8_to_lab_kernel and the fused frame ingest, which must agree bit for bit: keep the
// expressions here, in one place, so the compiler contracts them the same way in both.
__device__ __forceinline__ void rgb8_to_lab_px(const unsigned char px[3], float* L_out, float* A_out, float* B_out) {
  double c[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const double v = (double)px[k] / 255.0;
    c[k] = v > 0.04045 ? pow((v + 0.055) / 1.055, 2.4) : v / 12.92;
  }
  const double M[9] = {0.412453, 0.357580, 0.180423, 0.212671, 0.715160, 0.072169, 0.019334, 0.119193, 0.950227};
  const double white[3] = {0.95047, 1.0, 1.08883};
  double f[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const double t = (c[0] * M[k * 3 + 0] + c[1] * M[k * 3 + 1] + c[2] * M[k * 3 + 2]) / white[k];
    f[k] = t > 0.008856 ? cbrt(t) : 7.787 * t + 16.0 / 116.0;
  }
  const float L = (float)(116.0 * f[1] - 16.0), A = (float)(500.0 * (f[0] - f[1])), Bq = (float)(200.0 * (f[1] - f[2]));
  *L_out = L - 50.0f;
  *A_out = A;
  *B_out = Bq;
}
#endif

struct Act {
  float* d = nullptr;   // pixel (b=0, yp=0, xp=0), channel 0; the hi plane when lo != nullptr
  float* lo = nullptr;  // lo plane of a tf32 hi/lo split activation (value = hi + lo), same geometry
  // fp16 hi/lo planes of value * 2^e16 (same geometry, 2-byte elements); the fp32 plane `d` may coexist (d != nullptr)
  void* h16 = nullptr;
  void* l16 = nullptr;
  int e16 = 0;
  ScaleCell* cell = nullptr;  // set: e16 is unused, the exponent (and max |value|) live on the device
  int B = 0, H = 0, W = 0, C = 0, P = 0;
  int Hp() const { return H + 2 * P; }
  int Wp() const { return W + 2 * P; }
  size_t pixels() const { return (size_t)B * Hp() * Wp(); }
  size_t elems() const { return pixels() * C; }
};

enum ActFn { ACT_NONE = 0, ACT_RELU = 1, ACT_LRELU = 2 };
enum PadMode { PAD_ZERO = 0, PAD_REFLECT = 1 };

// ---- convolution as flat shifted GEMM --------------------------------------------------------
struct ConvParams {
  const float* x;  // input activation (padded NHWC)
  int Hp, Wp, P, H, W, Cin;
  const float* w;     // [taps][Cin][CoutPad]
  const float* bias;  // [CoutPad] (zeros beyond Cout) or nullptr
  int taps, dil, Cout, CoutPad, stride;
  int Ho, Wo;
  float* y;     // destination padded NHWC (interior written) or nullptr
  float* y_lo;  // when set, the value is stored as tf32 hi/lo planes (y = hi plane)
  int yHp, yWp, yP, yC, yCoff;
  const float* add;  // optional addend with the output's logical size (skip connections)
  int aHp, aWp, aP, aC;
  float* nchw;  // optional second destination [B][Cout][Ho][Wo]
  int act;
  float slope;
  double* stats;  // optional [B][Cout][2] (sum, sum of squares) of the stored values
  DynOut dyn;     // fp16 output planes with a device-derived scale (first layers in tensor-core mode)
};

void launch_conv_simt(const ConvParams& p, int B, bool two_level, cudaStream_t s);
// first layers (Cin padded to 8): one thread per output pixel; returns false if the shape is not covered
bool launch_conv_first(const ConvParams& p, int B, int cin_real, cudaStream_t s);

// ---- elementwise gather: InstanceNorm apply / PReLU / pad / up / sub / residual ----------------
struct XformParams {
  const float* src;
  const float* src_lo;  // optional lo plane of a split source
  int sH, sW, sP, sC, sCoff;
  float* dst;
  float* dst_lo;  // optional: store as hi/lo planes
  void* dst_h16;  // optional fp16 hi/lo planes of value * dscale16 (dst may be nullptr then)
  void* dst_l16;
  float dscale16;
  const float* res_lo;
  int dH, dW, dP, dC, dCoff;
  int C;
  int pad_mode, up, sub, rowpad;
  const double* stats;  // [B][C][2] or nullptr (no normalisation)
  double count;
  float eps;
  const float* scale;  // per-channel multiplier or nullptr
  const float* res;    // residual (padded NHWC, same logical size as dst) or nullptr
  int rP, rC;
  int act;  // 0 none, 1 relu, 2 prelu(slope)
  float slope;
};
void launch_xform(const XformParams& p, int B, cudaStream_t s);

// ---- per-pixel channel L2 normalisation (feature_normalize, theta/phi) --------------------------
struct PixNormParams {
  const float* src;
  const float* src_lo;
  const void* src_h16;  // fp16 hi/lo source planes of value * 2^(src_cell->e) (src may be nullptr then)
  const void* src_l16;
  const ScaleCell* src_cell;
  int sH, sW, sP, sC;
  float* dst;
  float* dst_lo;
  void* dst_h16;  // optional fp16 hi/lo planes of value * dscale16
  void* dst_l16;
  float dscale16;
  int dP, dC;  // destination has the same logical HxW
  int C, pad_mode;
  const double* stats;  // optional channel sums [B][C][2] -> subtract mean over positions
  double count;
  float eps;
};
void launch_pixnorm(const PixNormParams& p, int B, cudaStream_t s);

// ---- small layout / helper kernels -------------------------------------------------------------
// NCHW [B][Cs][H][W] -> padded NHWC with C channels (extra channels zero); mode: 0 copy,
// 1 rgb -> vgg_preprocess (util.py:347-352), 2 centred L -> gray -> vgg_preprocess (util.py:97-101),
// 3 centred Lab -> sRGB (util.py:379-414) -> vgg_preprocess
void launch_nchw_to_act(const float* src, int Cs, float* dst, float* dst_lo, int B, int H, int W, int C, int P,
                        int pad_mode, int mode, cudaStream_t s);
void launch_act_to_nchw(const float* src, const float* src_lo, int H, int W, int P, int sC, int sCoff, int C, float* dst,
                        int B, cudaStream_t s);
void launch_maxpool2(const float* src, const float* src_lo, int sH, int sW, int sP, int C, float* dst, float* dst_lo,
                     int dP, int B, cudaStream_t s);
// the same two on fp16 hi/lo planes with a device-side exponent (cell_out := cell_in for the pool: max-pooling
// non-negative values keeps both the scale and the max)
void launch_act_to_nchw_h16(const void* h16, const void* l16, const ScaleCell* cell, int H, int W, int P, int sC, int C,
                            float* dst, int B, cudaStream_t s);
void launch_maxpool2_h16(const void* h16, const void* l16, const ScaleCell* cell_in, int sH, int sW, int sP, int C,
                         void* dh16, void* dl16, ScaleCell* cell_out, int dP, int B, cudaStream_t s);
// max |x| over n floats -> cell->amax_bits (cell zeroed by the caller's arena)
void launch_amax(const float* x, size_t n, ScaleCell* cell, cudaStream_t s);
// NCHW [B][3][H][W] -> V [B][H/4*W/4][4] (4th lane ONE, see corr_tc.cu): F.avg_pool2d(.,4), NonlocalNet.py:491-493
void launch_avgpool4_lab(const float* src, float* V, int B, int H, int W, cudaStream_t s);
// rows [n][3] -> [n][4] = (x, y, z, 1); src == nullptr: only set the 4th lane of dst's rows to 1
void launch_pack_v4(const float* src3, float* dst4, size_t n, cudaStream_t s);
// y rows [B][N][4], sim rows [B][N] at h x w -> nearest x4 NCHW (NonlocalNet.py:499-500)
void launch_rows_to_nchw_up4(const float* yrows, const float* simrows, float* y, float* sim, int B, int h, int w,
                             cudaStream_t s);
// ColorVidNet input (FrameColor.py:64): [L, warped a, warped b, sim, last L, last a, last b, 0]
void launch_build_color_input(const float* IA_l, const float* yrows, const float* simrows, const float* last_lab,
                              float* dst, int B, int H, int W, int P, cudaStream_t s);
// conv10_ab (1x1, 128 -> 2) + tanh * 128 (ColorVidNet.py:143-144) -> NCHW [B][2][H][W]
void launch_final_ab(const float* x, int H, int W, int P, int C, const float* w /*[2][C]*/, const float* bias,
                     float* out, int B, cudaStream_t s);
// next frame's "last" = cat(L, ab) (test.py:96)
void launch_make_last(const float* IA_l, const float* ab, float* last, int B, int H, int W, cudaStream_t s);

// ---- correlation + softmax + warp (K7) ----------------------------------------------------------
// Peer outputs of a query-row-sharded correlation (SURVEY.md 8e, config 4): the rank that owns query rows
// [row0, row0 + NA) stores its result rows straight into the full-size result buffers of every GPU of the box
// (peer-mapped device pointers over NVLink) from the kernel that finalises them -- the all-gather IS the epilogue.
struct CorrPeers {
  int n = 0;           // number of destination GPUs (0: off)
  long long row0 = 0;  // global index of this rank's first query row
  float* y4[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};   // [N_total][4] each
  float* sim[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};  // [N_total] each
};

struct CorrParams {
  const float* theta;  // [B][NA][C]  (position-major, channels contiguous)
  const float* phi;    // [Bphi][NB][C]
  const float* V;      // [Bphi][NB][4] = (L, a, b, 1)
  int B, Bphi, NA, NB, C;
  float temperature;
  float* y;     // [B][NA][4]
  float* sim;   // [B][NA]
  int* argmax;  // [B][NA] or nullptr
  CorrPeers peers;  // optional fused all-gather of (y, sim) rows (B = 1 only)
  // tensor-core kernels only: per-query-row exponent scale log2(e) / T_i (forces the softmax epilogue, `temperature` is
  // ignored) and the softmax denominators sum_j exp((f_ij - max_j f_ij) / T_i) -- the contextual loss (ContextualLoss.py:115-126)
  const float* row_scale = nullptr;  // [B][NA]
  float* denom = nullptr;            // [B][NA]
};
// contextual-loss helpers (prepost.cu): channel means over positions, centred + L2-normalised position-major rows,
// per-row exponent scales from the row maxima, the final -log(mean_i 1 / denom_i)
void launch_chan_mean(const float* x, float* mean, int B, int C, int N, cudaStream_t s);
void launch_center_norm_rows(const float* x, const float* mean, float* rows, int B, int C, int N, float eps, cudaStream_t s);
void launch_ctx_row_scale(const float* rowmax, float* row_sc, size_t n, float h, cudaStream_t s);
void launch_ctx_loss(const float* denom, float* loss, int B, int N, cudaStream_t s);
void launch_corr_simt(const CorrParams& p, cudaStream_t s);
// [B][C][N] -> [B][N][C] and back (the C ABI of the stand-alone correlation entry is channel-major)
void launch_transpose_cn(const float* src, float* dst, int B, int C, int N, cudaStream_t s);

// pre / post-processing around the nets (test.py:58,71 and 100-102)
void launch_resize_half(const float* src, float* dst, int planes, int H, int W, cudaStream_t s);
void launch_upsample2(const float* src, float* dst, int planes, int h, int w, float scale, cudaStream_t s);
// sRGB uint8 HWC -> centred Lab NCHW fp32 (skimage.color.rgb2lab semantics in float64, then L - 50)
void launch_rgb8_to_lab(const unsigned char* rgb, float* lab, int B, int H, int W, cudaStream_t s);
// Lab -> sRGB uint8 HWC in float64 (skimage.color.lab2rgb semantics); rgb_from_xyz: row-major 3x3
void launch_lab_to_rgb8(const float* l, const float* ab, unsigned char* rgb, int B, int H, int W, const double* rgb_from_xyz,
                        cudaStream_t s);

// Fast Global Smoother (test.py:105-112) and the CenterPad resize (util_distortion.py:217-258): prepost.cu
// F frames: guides [F][H][W] -> weights [F][H][W]; the sweeps filter `planes` planes in place, every `ppg` consecutive planes
// guided by the weights of one frame
void launch_fgs_weights(const unsigned char* guide, const float* lut, float* Ch, float* Cv, int F, int H, int W, cudaStream_t s);
void launch_fgs_horizontal(float* cur, const float* Ch, float* D, int planes, int ppg, int H, int W, float lam, cudaStream_t s);
void launch_fgs_vertical(float* cur, const float* Cv, float* D, int planes, int ppg, int H, int W, float lam, cudaStream_t s);
void launch_l_to_guide8(const float* l, unsigned char* g, size_t n, cudaStream_t s);
void launch_gauss_axis_u8(const unsigned char* src, double* dst, const double* w, int radius, size_t n_outer, int len, int inner,
                          cudaStream_t s);
void launch_gauss_axis_f64(const double* src, double* dst, const double* w, int radius, size_t n_outer, int len, int inner,
                           cudaStream_t s);
void launch_zoom_crop(const double* src, int Hs, int Ws, int Hr, int Wr, int oy, int ox, unsigned char* dst, int Ho, int Wo,
                      cudaStream_t s);
// F anti-aliased float64 frames [F][Hs][Ws][3] -> zoom + crop / pad -> uint8 -> centred L [F][Ho][Wo] in one pass
void launch_ingest_l(const double* src, int F, int Hs, int Ws, int Hr, int Wr, int oy, int ox, float* l, int Ho, int Wo, cudaStream_t s);

int64_t launch_counter_add(int64_t n);  // global launch counter (introspection)

}  // namespace dvc
