// Pre / post-processing around the networks that the reference runs on the CPU (SURVEY.md §8f rows 2-3):
//
//  * Fast Global Smoother (the "WLS filter" of test.py:105-112: cv2.ximgproc.createFastGlobalSmootherFilter(guide,
//    lambda, sigma_color).filter(plane)).  Restated from Min, Choi, Lu, Ham, Sohn, Do, "Fast Global Image Smoothing Based
//    on Weighted Least Squares", IEEE TIP 2014 and the documented parameters of the OpenCV-contrib implementation
//    (lambda_attenuation = 0.25, num_iter = 3): per iteration one horizontal and one vertical sweep, each solving the
//    tridiagonal system  (I + lambda_n L) u = f  of every line with the Thomas algorithm in fp32, where L is the 1-D
//    graph Laplacian with weights exp(-|g_p - g_q| / sigma_color) between neighbours of the uint8 guide, and
//    lambda_{n+1} = lambda_n * lambda_attenuation.  opencv-contrib is not in this image: parity unpinned
//    (oracle/prepost_oracle.py restates the same algorithm and is validated against a float64 sparse solve).
//    HBM/latency-bound: the recurrences are sequential along a line, parallel across lines and planes.
//
//  * CenterPad (utils/util_distortion.py:217-258): aspect-preserving skimage.transform.resize(order=1, mode="reflect",
//    anti_aliasing=True, preserve_range=True, clip=False) -- i.e. scipy.ndimage.gaussian_filter(sigma = (factor-1)/2,
//    mode="mirror", truncate=4) followed by scipy.ndimage.zoom(order=1, mode="mirror", grid_mode=True), both float64 --
//    truncation to uint8 and the centred crop / zero pad to the target size.
#include <math.h>
#include <stdint.h>

#include "dvc_internal.cuh"

namespace dvc {

namespace {

// ------------------------------------------------------------------------------------------------ FGS
// C_h(i, j) = -w(g(i, j), g(i, j+1)), 0 in the last column; C_v(i, j) = -w(g(i, j), g(i+1, j)), 0 in the last row.
// F frames: guides [F][H][W] -> weights [F][H][W].
__global__ void __launch_bounds__(256) fgs_weights_kernel(const unsigned char* __restrict__ g, const float* __restrict__ lut,
                                                          float* __restrict__ Ch, float* __restrict__ Cv, int F, int H, int W) {
  const size_t hw = (size_t)H * W, n = (size_t)F * hw;
  for (size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x; p < n; p += (size_t)gridDim.x * blockDim.x) {
    const int q = (int)(p % hw);
    const int i = q / W, j = q - i * W;
    const int c = g[p];
    Ch[p] = (j + 1 < W) ? __ldg(lut + abs(c - (int)g[p + 1])) : 0.f;
    Cv[p] = (i + 1 < H) ? __ldg(lut + abs(c - (int)g[p + W])) : 0.f;
  }
}

// One line of the Thomas algorithm, element j of a line lives at base + j * stride.  Every operation is a separately
// rounded fp32 operation (no FMA contraction), in the order of the oracle.
//   forward : denom_j = (1 - lam C_{j-1} - lam C_j) - lam C_{j-1} * D_{j-1};  D_j = lam C_j / denom_j;
//             u_j = (u_j - lam C_{j-1} u_{j-1}) / denom_j
//   backward: u_j = u_j - D_j u_{j+1}
// Both sweeps take `planes` planes of which every `ppg` consecutive ones share one guide (plane pl uses the weights of
// frame pl / ppg): one launch covers all planes of all frames.
// Vertical sweep: thread = (plane, column), adjacent threads touch adjacent addresses (coalesced); one grid row per frame.
__global__ void __launch_bounds__(128) fgs_vertical_kernel(float* __restrict__ cur, const float* __restrict__ Cv, float* __restrict__ D,
                                                           int ppg, int H, int W, float lam) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;  // blockIdx.y = frame
  if (t >= ppg * W) return;
  const int pl = blockIdx.y * ppg + t / W, x = t % W;
  float* u = cur + (size_t)pl * H * W + x;
  float* d = D + (size_t)pl * H * W + x;
  const float* c = Cv + (size_t)blockIdx.y * H * W + x;
  float cprev = __fmul_rn(lam, c[0]);
  float denom = __fsub_rn(1.f, cprev);
  float dprev = __fdiv_rn(cprev, denom);
  float uprev = __fdiv_rn(u[0], denom);
  d[0] = dprev, u[0] = uprev;
  for (int i = 1; i < H; ++i) {
    const float ci = __fmul_rn(lam, c[(size_t)i * W]);
    denom = __fsub_rn(__fsub_rn(__fsub_rn(1.f, cprev), ci), __fmul_rn(cprev, dprev));
    dprev = __fdiv_rn(ci, denom);
    uprev = __fdiv_rn(__fsub_rn(u[(size_t)i * W], __fmul_rn(cprev, uprev)), denom);
    d[(size_t)i * W] = dprev, u[(size_t)i * W] = uprev;
    cprev = ci;
  }
  for (int i = H - 2; i >= 0; --i) {
    uprev = __fsub_rn(u[(size_t)i * W], __fmul_rn(d[(size_t)i * W], uprev));
    u[(size_t)i * W] = uprev;
  }
}

// Horizontal sweep: one warp owns 32 consecutive rows of one plane (lane = row) and walks along x in 32-column tiles
// that are moved between global and shared memory with coalesced row accesses (a thread per row reading its own row
// directly would touch one sector per element).
__global__ void __launch_bounds__(32) fgs_horizontal_kernel(float* __restrict__ cur, const float* __restrict__ Ch, float* __restrict__ D,
                                                            int planes, int ppg, int H, int W, float lam) {
  __shared__ float su[32][33], sc[32][33], sd[32][33];
  const int lane = threadIdx.x;
  const int groups = (H + 31) / 32;
  const int pl = blockIdx.x / groups, r0 = (blockIdx.x - pl * groups) * 32;
  const int nrows = min(32, H - r0);
  float* ub = cur + ((size_t)pl * H + r0) * W;
  float* db = D + ((size_t)pl * H + r0) * W;
  const float* cb = Ch + ((size_t)(pl / ppg) * H + r0) * W;
  float cprev = 0.f, dprev = 0.f, uprev = 0.f;
  for (int x0 = 0; x0 < W; x0 += 32) {
    const int nx = min(32, W - x0);
    for (int k = 0; k < nrows; ++k)
      if (lane < nx) su[k][lane] = ub[(size_t)k * W + x0 + lane], sc[k][lane] = __ldg(cb + (size_t)k * W + x0 + lane);
    __syncwarp();
    if (lane < nrows) {
      for (int j = 0; j < nx; ++j) {
        const float cj = __fmul_rn(lam, sc[lane][j]);
        float denom;
        if (x0 + j == 0)
          denom = __fsub_rn(1.f, cj);
        else
          denom = __fsub_rn(__fsub_rn(__fsub_rn(1.f, cprev), cj), __fmul_rn(cprev, dprev));
        dprev = __fdiv_rn(cj, denom);
        uprev = (x0 + j == 0) ? __fdiv_rn(su[lane][j], denom) : __fdiv_rn(__fsub_rn(su[lane][j], __fmul_rn(cprev, uprev)), denom);
        sd[lane][j] = dprev, su[lane][j] = uprev;
        cprev = cj;
      }
    }
    __syncwarp();
    for (int k = 0; k < nrows; ++k)
      if (lane < nx) ub[(size_t)k * W + x0 + lane] = su[k][lane], db[(size_t)k * W + x0 + lane] = sd[k][lane];
    __syncwarp();
  }
  // backward substitution, tiles right to left; uprev holds u_{W-1}
  const int last_tile = ((W - 1) / 32) * 32;
  for (int x0 = last_tile; x0 >= 0; x0 -= 32) {
    const int nx = min(32, W - x0);
    for (int k = 0; k < nrows; ++k)
      if (lane < nx) su[k][lane] = ub[(size_t)k * W + x0 + lane], sd[k][lane] = db[(size_t)k * W + x0 + lane];
    __syncwarp();
    if (lane < nrows) {
      for (int j = nx - 1; j >= 0; --j) {
        if (x0 + j == W - 1) continue;  // u_{W-1} is final after the forward sweep
        uprev = __fsub_rn(su[lane][j], __fmul_rn(sd[lane][j], uprev));
        su[lane][j] = uprev;
      }
    }
    __syncwarp();
    for (int k = 0; k < nrows; ++k)
      if (lane < nx) ub[(size_t)k * W + x0 + lane] = su[k][lane];
    __syncwarp();
  }
}

// test.py:106: guide = uint8(uncenter_l(L) * 255 / 100), fp32 arithmetic, truncation toward zero
__global__ void __launch_bounds__(256) l_to_guide8_kernel(const float* __restrict__ l, unsigned char* __restrict__ g, size_t n) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const float v = __fdiv_rn(__fmul_rn(__fadd_rn(__ldg(l + i), 50.f), 255.f), 100.f);
    g[i] = (unsigned char)fminf(fmaxf(truncf(v), 0.f), 255.f);
  }
}

// ------------------------------------------------------------------------------------------------ CenterPad resize
__device__ __forceinline__ int mirror_idx(int i, int n) {  // scipy.ndimage mode="mirror": d c b | a b c d | c b a
  if (n == 1) return 0;
  const int period = 2 * (n - 1);
  i = i % period;
  if (i < 0) i += period;
  return i < n ? i : period - i;
}

// Gaussian along one axis in float64 (scipy.ndimage.gaussian_filter1d: weights exp(-0.5 k^2 / sigma^2) / sum, radius
// int(4 sigma + 0.5), correlate with mode="mirror").  src [n_outer][len][inner] -> dst, taps in `w` (2 r + 1 doubles).
template <typename TIn>
__global__ void __launch_bounds__(256) gauss_axis_kernel(const TIn* __restrict__ src, double* __restrict__ dst, const double* __restrict__ w,
                                                         int radius, size_t n_outer, int len, int inner) {
  const size_t total = n_outer * (size_t)len * inner;
  for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const int in_i = (int)(idx % inner);
    const size_t t = idx / inner;
    const int pos = (int)(t % len);
    const size_t outer = t / len;
    const TIn* base = src + outer * (size_t)len * inner + in_i;
    // scipy's correlate1d for symmetric weights: centre tap first, then the pairs (left + right) * w from the OUTSIDE in.
    // Separately rounded multiplies and adds (no FMA contraction): with sigma = 0.125 (a 1.25x down-scale) the taps are
    // (1.3e-14, 1, 1.3e-14), the filtered values sit within 1e-12 of integers and the final truncation to uint8 sees
    // the last bit -- scipy's C code is compiled without FMA.
    double acc = __dmul_rn((double)base[(size_t)pos * inner], w[radius]);
    for (int k = radius; k >= 1; --k) {
      const double l = (double)base[(size_t)mirror_idx(pos - k, len) * inner], r = (double)base[(size_t)mirror_idx(pos + k, len) * inner];
      acc = __dadd_rn(acc, __dmul_rn(__dadd_rn(l, r), w[radius + k]));
    }
    dst[idx] = acc;
  }
}

// scipy.ndimage.zoom(order=1, mode="mirror", grid_mode=True) of a [Hs][Ws][3] float64 image to [Hr][Wr], channel ch of
// resized pixel (yr, xr), truncated to uint8 (ndarray.astype(np.uint8) of in-range values).
__device__ __forceinline__ unsigned char zoom_px(const double* __restrict__ src, int Hs, int Ws, int Hr, int Wr, int yr, int xr, int ch) {
  // grid_mode: pixel centres align, in = (out + 0.5) * (in_len / out_len) - 0.5
  // (separately rounded operations throughout: see gauss_axis_kernel)
  const double cy = __dsub_rn(__dmul_rn(__dadd_rn((double)yr, 0.5), __ddiv_rn((double)Hs, (double)Hr)), 0.5);
  const double cx = __dsub_rn(__dmul_rn(__dadd_rn((double)xr, 0.5), __ddiv_rn((double)Ws, (double)Wr)), 0.5);
  const double fy = floor(cy), fx = floor(cx);
  const double ty = __dsub_rn(cy, fy), tx = __dsub_rn(cx, fx);
  const int y0 = mirror_idx((int)fy, Hs), y1 = mirror_idx((int)fy + 1, Hs);
  const int x0 = mirror_idx((int)fx, Ws), x1 = mirror_idx((int)fx + 1, Ws);
  const double v00 = src[((size_t)y0 * Ws + x0) * 3 + ch], v01 = src[((size_t)y0 * Ws + x1) * 3 + ch];
  const double v10 = src[((size_t)y1 * Ws + x0) * 3 + ch], v11 = src[((size_t)y1 * Ws + x1) * 3 + ch];
  // scipy (ni_interpolation.c) sums the 2 x 2 neighbourhood, row-major, each term ((value * wy) * wx)
  const double wy0 = __dsub_rn(1.0, ty), wx0 = __dsub_rn(1.0, tx);
  double v = __dmul_rn(__dmul_rn(v00, wy0), wx0);
  v = __dadd_rn(v, __dmul_rn(__dmul_rn(v01, wy0), tx));
  v = __dadd_rn(v, __dmul_rn(__dmul_rn(v10, ty), wx0));
  v = __dadd_rn(v, __dmul_rn(__dmul_rn(v11, ty), tx));
  return (unsigned char)fmin(fmax(trunc(v), 0.0), 255.0);
}

// zoom_px, then CenterPad's centred crop (offset oy, ox) / zero pad into the [Ho][Wo][3] output.
__global__ void __launch_bounds__(256) zoom_crop_kernel(const double* __restrict__ src, int Hs, int Ws, int Hr, int Wr, int oy, int ox,
                                                        unsigned char* __restrict__ dst, int Ho, int Wo) {
  const size_t total = (size_t)Ho * Wo * 3;
  for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const int ch = (int)(idx % 3);
    const size_t t = idx / 3;
    const int xo = (int)(t % Wo), yo = (int)(t / Wo);
    const int yr = yo + oy, xr = xo + ox;  // position in the resized image
    dst[idx] = (yr >= 0 && yr < Hr && xr >= 0 && xr < Wr) ? zoom_px(src, Hs, Ws, Hr, Wr, yr, xr, ch) : 0;
  }
}

// The frame ingest of test.py:44-46 after the anti-aliasing Gaussians, for F frames [F][Hs][Ws][3] float64: zoom + crop /
// pad (zoom_crop_kernel) -> sRGB uint8 -> Lab (rgb8_to_lab_px) -> centred L [F][Ho][Wo].  The uint8 pixel never leaves
// registers; a/b are not needed by the networks' input and are not written.
__global__ void __launch_bounds__(256) ingest_l_kernel(const double* __restrict__ src, int F, int Hs, int Ws, int Hr, int Wr, int oy,
                                                       int ox, float* __restrict__ l, int Ho, int Wo) {
  const size_t hw = (size_t)Ho * Wo, total = (size_t)F * hw;
  for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const size_t f = idx / hw, q = idx - f * hw;
    const int xo = (int)(q % Wo), yo = (int)(q / Wo);
    const int yr = yo + oy, xr = xo + ox;
    const double* fs = src + f * (size_t)Hs * Ws * 3;
    unsigned char px[3] = {0, 0, 0};
    if (yr >= 0 && yr < Hr && xr >= 0 && xr < Wr) {
#pragma unroll
      for (int ch = 0; ch < 3; ++ch) px[ch] = zoom_px(fs, Hs, Ws, Hr, Wr, yr, xr, ch);
    }
    float L, A, Bq;
    rgb8_to_lab_px(px, &L, &A, &Bq);
    l[idx] = L;
  }
}

// ------------------------------------------------------------------------------------------------ contextual loss
// mean over the N positions of every (image, channel): one block per (b, c), double accumulation
__global__ void __launch_bounds__(256) chan_mean_kernel(const float* __restrict__ x, float* __restrict__ mean, int N) {
  __shared__ double red[256];
  const float* p = x + (size_t)blockIdx.x * N;
  double acc = 0.0;
  for (int i = threadIdx.x; i < N; i += 256) acc += (double)__ldg(p + i);
  red[threadIdx.x] = acc;
  __syncthreads();
  for (int o = 128; o >= 1; o >>= 1) {
    if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) mean[blockIdx.x] = (float)(red[0] / N);
}

// NCHW [B][C][N] -> position-major rows [B][N][C] of (x - mean_c) / (||x - mean||_2 over C + eps)  (ContextualLoss.py:99-111,
// feature_normalize util.py:155-158).  One block = 32 positions: first the norms (reads coalesced over positions), then a
// 32 x 32 shared-memory transpose per channel group so that the row stores are contiguous.
__global__ void __launch_bounds__(256) center_norm_rows_kernel(const float* __restrict__ x, const float* __restrict__ mean,
                                                               float* __restrict__ rows, int C, int N, float eps) {
  __shared__ float tile[32][33];
  __shared__ float s_inv[32];
  __shared__ float s_part[8][32];
  const int b = blockIdx.y, n0 = blockIdx.x * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
  const float* xb = x + (size_t)b * C * N;
  const float* mb = mean ? mean + (size_t)b * C : nullptr;
  const int n = n0 + tx;
  float ss = 0.f;
  for (int c = ty; c < C; c += 8) {
    const float v = (n < N ? __ldg(xb + (size_t)c * N + n) : 0.f) - (mb ? __ldg(mb + c) : 0.f);
    ss = fmaf(v, v, ss);
  }
  s_part[ty][tx] = ss;
  __syncthreads();
  if (ty == 0) {
    float t = 0.f;
    for (int k = 0; k < 8; ++k) t += s_part[k][tx];
    s_inv[tx] = 1.f / (sqrtf(t) + eps);
  }
  __syncthreads();
  for (int c0 = 0; c0 < C; c0 += 32) {
    for (int k = ty; k < 32; k += 8) {  // channel c0 + k, position n0 + tx
      const int c = c0 + k;
      tile[k][tx] = (c < C && n < N) ? (__ldg(xb + (size_t)c * N + n) - (mb ? __ldg(mb + c) : 0.f)) * s_inv[tx] : 0.f;
    }
    __syncthreads();
    for (int k = ty; k < 32; k += 8) {  // position n0 + k, channel c0 + tx
      if (n0 + k < N && c0 + tx < C) rows[((size_t)b * N + n0 + k) * C + c0 + tx] = tile[tx][k];
    }
    __syncthreads();
  }
}

// log2(e) / T_i with T_i = h * (min_j d_ij + 1e-5) = h * (1 - max_j f_ij + 1e-5)   (ContextualLoss.py:118-122)
__global__ void __launch_bounds__(256) ctx_row_scale_kernel(const float* __restrict__ rowmax, float* __restrict__ row_sc, size_t n, float h) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    row_sc[i] = 1.4426950408889634f / (h * ((1.f - __ldg(rowmax + i)) + 1e-5f));
}

// loss_b = -log(mean_i max_j A_ij) with max_j A_ij = 1 / sum_j exp((f_ij - m_i) / T_i)   (ContextualLoss.py:123-126)
__global__ void __launch_bounds__(256) ctx_loss_kernel(const float* __restrict__ denom, float* __restrict__ loss, int N) {
  __shared__ double red[256];
  const float* p = denom + (size_t)blockIdx.x * N;
  double acc = 0.0;
  for (int i = threadIdx.x; i < N; i += 256) acc += 1.0 / (double)__ldg(p + i);
  red[threadIdx.x] = acc;
  __syncthreads();
  for (int o = 128; o >= 1; o >>= 1) {
    if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) loss[blockIdx.x] = (float)(-log(red[0] / N));
}

inline int grid_for(size_t total, int threads, int cap = 148 * 16) {
  const size_t g = (total + threads - 1) / threads;
  return (int)(g < (size_t)cap ? (g ? g : 1) : cap);
}

}  // namespace

void launch_chan_mean(const float* x, float* mean, int B, int C, int N, cudaStream_t s) {
  chan_mean_kernel<<<B * C, 256, 0, s>>>(x, mean, N);
  launch_counter_add(1);
}
void launch_center_norm_rows(const float* x, const float* mean, float* rows, int B, int C, int N, float eps, cudaStream_t s) {
  center_norm_rows_kernel<<<dim3((N + 31) / 32, B), 256, 0, s>>>(x, mean, rows, C, N, eps);
  launch_counter_add(1);
}
void launch_ctx_row_scale(const float* rowmax, float* row_sc, size_t n, float h, cudaStream_t s) {
  ctx_row_scale_kernel<<<grid_for(n, 256), 256, 0, s>>>(rowmax, row_sc, n, h);
  launch_counter_add(1);
}
void launch_ctx_loss(const float* denom, float* loss, int B, int N, cudaStream_t s) {
  ctx_loss_kernel<<<B, 256, 0, s>>>(denom, loss, N);
  launch_counter_add(1);
}
void launch_fgs_weights(const unsigned char* guide, const float* lut, float* Ch, float* Cv, int F, int H, int W, cudaStream_t s) {
  fgs_weights_kernel<<<grid_for((size_t)F * H * W, 256), 256, 0, s>>>(guide, lut, Ch, Cv, F, H, W);
  launch_counter_add(1);
}
void launch_fgs_horizontal(float* cur, const float* Ch, float* D, int planes, int ppg, int H, int W, float lam, cudaStream_t s) {
  fgs_horizontal_kernel<<<planes * ((H + 31) / 32), 32, 0, s>>>(cur, Ch, D, planes, ppg, H, W, lam);
  launch_counter_add(1);
}
void launch_fgs_vertical(float* cur, const float* Cv, float* D, int planes, int ppg, int H, int W, float lam, cudaStream_t s) {
  fgs_vertical_kernel<<<dim3((ppg * W + 127) / 128, planes / ppg), 128, 0, s>>>(cur, Cv, D, ppg, H, W, lam);
  launch_counter_add(1);
}
void launch_l_to_guide8(const float* l, unsigned char* g, size_t n, cudaStream_t s) {
  l_to_guide8_kernel<<<grid_for(n, 256), 256, 0, s>>>(l, g, n);
  launch_counter_add(1);
}
void launch_gauss_axis_u8(const unsigned char* src, double* dst, const double* w, int radius, size_t n_outer, int len, int inner,
                          cudaStream_t s) {
  gauss_axis_kernel<unsigned char><<<grid_for(n_outer * len * inner, 256), 256, 0, s>>>(src, dst, w, radius, n_outer, len, inner);
  launch_counter_add(1);
}
void launch_gauss_axis_f64(const double* src, double* dst, const double* w, int radius, size_t n_outer, int len, int inner,
                           cudaStream_t s) {
  gauss_axis_kernel<double><<<grid_for(n_outer * len * inner, 256), 256, 0, s>>>(src, dst, w, radius, n_outer, len, inner);
  launch_counter_add(1);
}
void launch_zoom_crop(const double* src, int Hs, int Ws, int Hr, int Wr, int oy, int ox, unsigned char* dst, int Ho, int Wo,
                      cudaStream_t s) {
  zoom_crop_kernel<<<grid_for((size_t)Ho * Wo * 3, 256), 256, 0, s>>>(src, Hs, Ws, Hr, Wr, oy, ox, dst, Ho, Wo);
  launch_counter_add(1);
}
void launch_ingest_l(const double* src, int F, int Hs, int Ws, int Hr, int Wr, int oy, int ox, float* l, int Ho, int Wo, cudaStream_t s) {
  ingest_l_kernel<<<grid_for((size_t)F * Ho * Wo, 256), 256, 0, s>>>(src, F, Hs, Ws, Hr, Wr, oy, ox, l, Ho, Wo);
  launch_counter_add(1);
}

}  // namespace dvc
