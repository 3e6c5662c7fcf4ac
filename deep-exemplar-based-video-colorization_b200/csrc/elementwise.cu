// HBM-bound helper kernels around the GEMM-shaped ones: InstanceNorm apply / PReLU / padding /
// nearest up-sampling / stride-2 pick / residual add (one gather kernel), per-pixel channel
// normalisation, max-pool, layout conversion at the NCHW boundary, colour-space prologue.
// All are coalesced over the channel (innermost) dimension with 128-bit accesses.
#include <cuda_fp16.h>
#include <math.h>

#include "dvc_internal.cuh"

namespace dvc {

namespace {

__device__ __forceinline__ float tf32_rna(float x) {
  uint32_t u;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(x));
  return __uint_as_float(u);
}
// value of a (possibly hi/lo split) activation
__device__ __forceinline__ float4 ld4(const float* __restrict__ p, const float* __restrict__ lo, size_t off) {
  float4 v = __ldg(reinterpret_cast<const float4*>(p + off));
  if (lo) {
    const float4 l = __ldg(reinterpret_cast<const float4*>(lo + off));
    v.x += l.x, v.y += l.y, v.z += l.z, v.w += l.w;
  }
  return v;
}
// store as fp32, or as tf32 hi/lo planes for a tensor-core consumer (hi + lo reproduces v to 2^-24 relative)
__device__ __forceinline__ void st4(float* __restrict__ p, float* __restrict__ lo, size_t off, float4 v) {
  if (lo) {
    const float4 h = make_float4(tf32_rna(v.x), tf32_rna(v.y), tf32_rna(v.z), tf32_rna(v.w));
    *reinterpret_cast<float4*>(p + off) = h;
    *reinterpret_cast<float4*>(lo + off) =
        make_float4(tf32_rna(v.x - h.x), tf32_rna(v.y - h.y), tf32_rna(v.z - h.z), tf32_rna(v.w - h.w));
  } else {
    *reinterpret_cast<float4*>(p + off) = v;
  }
}

// fp16 hi/lo planes of v * scale (scale = 2^e from a proven bound on |v|, so the clamp never triggers in range):
// hi + lo carries 2 x 11 significant bits like the tf32 split, at half the bytes
__device__ __forceinline__ void st4h(__half* __restrict__ hp, __half* __restrict__ lp, size_t off, float4 v, float scale) {
  const float x[4] = {v.x * scale, v.y * scale, v.z * scale, v.w * scale};
  unsigned short h[4], l[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float xc = fminf(fmaxf(x[j], -65504.f), 65504.f);
    const __half hh = __float2half_rn(xc);
    h[j] = __half_as_ushort(hh);
    l[j] = __half_as_ushort(__float2half_rn(xc - __half2float(hh)));
  }
  *reinterpret_cast<uint2*>(hp + off) = make_uint2((uint32_t)h[0] | ((uint32_t)h[1] << 16), (uint32_t)h[2] | ((uint32_t)h[3] << 16));
  *reinterpret_cast<uint2*>(lp + off) = make_uint2((uint32_t)l[0] | ((uint32_t)l[1] << 16), (uint32_t)l[2] | ((uint32_t)l[3] << 16));
}

// 4 channels of an fp16 hi/lo activation, in scaled units (hi + lo is exact in fp32: 2 x 11 significant bits)
__device__ __forceinline__ float4 ld4h(const __half* __restrict__ hp, const __half* __restrict__ lp, size_t off) {
  const uint2 h = __ldg(reinterpret_cast<const uint2*>(hp + off)), l = __ldg(reinterpret_cast<const uint2*>(lp + off));
  const float2 h0 = __half22float2(*reinterpret_cast<const __half2*>(&h.x)), h1 = __half22float2(*reinterpret_cast<const __half2*>(&h.y));
  const float2 l0 = __half22float2(*reinterpret_cast<const __half2*>(&l.x)), l1 = __half22float2(*reinterpret_cast<const __half2*>(&l.y));
  return make_float4(h0.x + l0.x, h0.y + l0.y, h1.x + l1.x, h1.y + l1.y);
}

__device__ __forceinline__ int reflect_idx(int i, int n) {
  if (i < 0) i = -i;
  if (i >= n) i = 2 * (n - 1) - i;
  return i;
}

// ------------------------------------------------------------------------------------ xform
// dst-driven gather.  grid.y = image, grid.x covers (padded dst pixels) x (C/4) float4 lanes.
__global__ void __launch_bounds__(256) xform_kernel(const XformParams p) {
  extern __shared__ float sm[];  // mean[C], rstd[C] when normalising
  const int b = blockIdx.y;
  float* s_mean = sm;
  float* s_rstd = sm + p.C;
  if (p.stats) {
    for (int c = threadIdx.x; c < p.C; c += blockDim.x) {
      const double su = p.stats[((size_t)b * p.C + c) * 2 + 0];
      const double sq = p.stats[((size_t)b * p.C + c) * 2 + 1];
      const double mean = su / p.count;
      double var = sq / p.count - mean * mean;  // biased variance, F.instance_norm
      if (var < 0) var = 0;
      s_mean[c] = (float)mean;
      s_rstd[c] = (float)(1.0 / sqrt(var + (double)p.eps));
    }
    __syncthreads();
  }
  const int dHp = p.dH + 2 * p.dP, dWp = p.dW + 2 * p.dP;
  const int sWp = p.sW + 2 * p.sP, sHp = p.sH + 2 * p.sP;
  // one thread = 8 channels of one destination pixel; 32-bit index math (dHp * dWp * C / 8 < 2^31 by far)
  const int c8n = p.C >> 3;
  const int total = dHp * dWp * c8n;
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
    const int pix = idx / c8n;
    const int c = (idx - pix * c8n) * 8;
    const int yp = pix / dWp, xp = pix - yp * dWp;
    int y = yp - p.dP, x = xp - p.dP;
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = 0.f;
    bool inside = (y >= 0 && y < p.dH && x >= 0 && x < p.dW);
    if (!inside && p.pad_mode == PAD_REFLECT) {
      y = reflect_idx(y, p.dH);
      x = reflect_idx(x, p.dW);
      inside = true;
    }
    if (inside) {
      int y1 = y;
      if (p.rowpad) y1 = min(max(y - 1, 0), p.dH - 3);
      const int ys = (y1 / p.up) * p.sub, xs = (x / p.up) * p.sub;
      const size_t so = (((size_t)b * sHp + ys + p.sP) * sWp + xs + p.sP) * p.sC + p.sCoff + c;
      const float4 v0 = ld4(p.src, p.src_lo, so), v1 = ld4(p.src, p.src_lo, so + 4);
      v[0] = v0.x, v[1] = v0.y, v[2] = v0.z, v[3] = v0.w, v[4] = v1.x, v[5] = v1.y, v[6] = v1.z, v[7] = v1.w;
      if (p.stats) {
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = (v[j] - s_mean[c + j]) * s_rstd[c + j];
      }
      if (p.scale) {
        const float4 s0 = __ldg(reinterpret_cast<const float4*>(p.scale + c)), s1 = __ldg(reinterpret_cast<const float4*>(p.scale + c + 4));
        v[0] *= s0.x, v[1] *= s0.y, v[2] *= s0.z, v[3] *= s0.w, v[4] *= s1.x, v[5] *= s1.y, v[6] *= s1.z, v[7] *= s1.w;
      }
      if (p.res) {
        const int rHp = p.dH + 2 * p.rP, rWp = p.dW + 2 * p.rP;
        const size_t ro = (((size_t)b * rHp + y + p.rP) * rWp + x + p.rP) * p.rC + c;
        const float4 r0 = ld4(p.res, p.res_lo, ro), r1 = ld4(p.res, p.res_lo, ro + 4);
        v[0] += r0.x, v[1] += r0.y, v[2] += r0.z, v[3] += r0.w, v[4] += r1.x, v[5] += r1.y, v[6] += r1.z, v[7] += r1.w;
      }
      if (p.act == 1) {
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = fmaxf(v[j], 0.f);
      } else if (p.act == 2) {
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = v[j] > 0.f ? v[j] : v[j] * p.slope;
      }
    }
    const size_t doff = (((size_t)b * dHp + yp) * dWp + xp) * p.dC + p.dCoff + c;
    if (p.dst) {
      st4(p.dst, p.dst_lo, doff, make_float4(v[0], v[1], v[2], v[3]));
      st4(p.dst, p.dst_lo, doff + 4, make_float4(v[4], v[5], v[6], v[7]));
    }
    if (p.dst_h16) {
      uint32_t hw[4], lw[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float a0 = fminf(fmaxf(v[2 * j] * p.dscale16, -65504.f), 65504.f);
        const float a1 = fminf(fmaxf(v[2 * j + 1] * p.dscale16, -65504.f), 65504.f);
        const __half2 h2 = __floats2half2_rn(a0, a1);
        const float2 hf = __half22float2(h2);
        const __half2 l2 = __floats2half2_rn(a0 - hf.x, a1 - hf.y);
        hw[j] = *reinterpret_cast<const uint32_t*>(&h2), lw[j] = *reinterpret_cast<const uint32_t*>(&l2);
      }
      *reinterpret_cast<uint4*>(reinterpret_cast<__half*>(p.dst_h16) + doff) = make_uint4(hw[0], hw[1], hw[2], hw[3]);
      *reinterpret_cast<uint4*>(reinterpret_cast<__half*>(p.dst_l16) + doff) = make_uint4(lw[0], lw[1], lw[2], lw[3]);
    }
  }
}

// ------------------------------------------------------------------------------------ pixnorm
// One warp per destination (padded) pixel: out = (v - mean_c) / (||v - mean||_2 + eps).
template <int VPL>  // float4 per lane: C = 128 * VPL
__global__ void __launch_bounds__(256) pixnorm_kernel(const PixNormParams p) {
  const int b = blockIdx.y;
  const int lane = threadIdx.x & 31;
  const int dHp = p.sH + 2 * p.dP, dWp = p.sW + 2 * p.dP;
  const int sHp = p.sH + 2 * p.sP, sWp = p.sW + 2 * p.sP;
  const int warps_per_grid = gridDim.x * (blockDim.x >> 5);
  const float descale = p.src_h16 ? exp2_int(-p.src_cell->e) : 1.f;
  float4 mean[VPL];
#pragma unroll
  for (int i = 0; i < VPL; ++i) {
    mean[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (p.stats) {
      const int c = (i * 32 + lane) * 4;
      const double* st = p.stats + ((size_t)b * p.C + c) * 2;
      mean[i] = make_float4((float)(st[0] / p.count), (float)(st[2] / p.count), (float)(st[4] / p.count),
                            (float)(st[6] / p.count));
    }
  }
  for (int pix = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); pix < dHp * dWp; pix += warps_per_grid) {
    const int yp = pix / dWp, xp = pix - yp * dWp;
    int y = yp - p.dP, x = xp - p.dP;
    bool inside = (y >= 0 && y < p.sH && x >= 0 && x < p.sW);
    if (!inside && p.pad_mode == PAD_REFLECT) {
      y = reflect_idx(y, p.sH);
      x = reflect_idx(x, p.sW);
      inside = true;
    }
    float4 v[VPL];
    float ss = 0.f;
    const size_t so = (((size_t)b * sHp + y + p.sP) * sWp + x + p.sP) * p.sC;
#pragma unroll
    for (int i = 0; i < VPL; ++i) {
      if (inside) {
        if (p.src_h16) {
          v[i] = ld4h(reinterpret_cast<const __half*>(p.src_h16), reinterpret_cast<const __half*>(p.src_l16), so + (i * 32 + lane) * 4);
          v[i].x *= descale, v[i].y *= descale, v[i].z *= descale, v[i].w *= descale;
        } else {
          v[i] = ld4(p.src, p.src_lo, so + (i * 32 + lane) * 4);
        }
        v[i].x -= mean[i].x, v[i].y -= mean[i].y, v[i].z -= mean[i].z, v[i].w -= mean[i].w;
      } else {
        v[i] = make_float4(0.f, 0.f, 0.f, 0.f);
      }
      ss += v[i].x * v[i].x + v[i].y * v[i].y + v[i].z * v[i].z + v[i].w * v[i].w;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
    const size_t dof = (((size_t)b * dHp + yp) * dWp + xp) * p.dC;
    const float n = sqrtf(ss) + p.eps;
#pragma unroll
    for (int i = 0; i < VPL; ++i) {
      // true division like torch.div(x, norm) (util.py:157, NonlocalNet.py:471)
      const float4 o4 = make_float4(v[i].x / n, v[i].y / n, v[i].z / n, v[i].w / n);
      if (p.dst) st4(p.dst, p.dst_lo, dof + (i * 32 + lane) * 4, o4);
      if (p.dst_h16)
        st4h(reinterpret_cast<__half*>(p.dst_h16), reinterpret_cast<__half*>(p.dst_l16), dof + (i * 32 + lane) * 4, o4, p.dscale16);
    }
  }
}

// ------------------------------------------------------------------------------------ colour prologue
__device__ __forceinline__ float3 lab_to_srgb(float L, float a, float bb) {
  // util.py:379-414 (L un-centred)
  float fy = (L + 16.0f) / 116.0f;
  float fx = a / 500.0f + fy;
  float fz = fy - bb / 200.0f;
  if (fz < 0.f) fz = 0.f;
  float f[3] = {fx, fy, fz};
  float lin[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) lin[i] = f[i] > 0.2068966f ? powf(f[i], 3.0f) : (f[i] - 16.0f / 116.0f) / 7.787f;
  lin[0] *= 0.95047f;
  lin[2] *= 1.08883f;
  const float m[3][3] = {{3.24048134f, -0.96925495f, 0.05564664f},
                         {-1.53715152f, 1.87599f, -0.20404134f},
                         {-0.49853633f, 0.04155593f, 1.05731107f}};
  float rgb[3];
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    float r = lin[0] * m[0][j];
    r = fmaf(lin[1], m[1][j], r);
    r = fmaf(lin[2], m[2][j], r);
    r = r > 0.0031308f ? 1.055f * powf(r, 1.0f / 2.4f) - 0.055f : r * 12.92f;
    rgb[j] = fminf(fmaxf(r, 0.f), 1.f);
  }
  return make_float3(rgb[0], rgb[1], rgb[2]);
}

__global__ void __launch_bounds__(256) nchw_to_act_kernel(const float* __restrict__ src, int Cs, float* __restrict__ dst,
                                                          float* __restrict__ dst_lo, int H, int W, int C, int P,
                                                          int pad_mode, int mode) {
  const int b = blockIdx.y;
  const int Hp = H + 2 * P, Wp = W + 2 * P;
  const size_t plane = (size_t)H * W;
  for (int pix = blockIdx.x * blockDim.x + threadIdx.x; pix < Hp * Wp; pix += gridDim.x * blockDim.x) {
    const int yp = pix / Wp, xp = pix - yp * Wp;
    int y = yp - P, x = xp - P;
    bool inside = (y >= 0 && y < H && x >= 0 && x < W);
    if (!inside && pad_mode == PAD_REFLECT) {
      y = reflect_idx(y, H), x = reflect_idx(x, W);
      inside = true;
    }
    float* dp = dst + ((size_t)b * Hp * Wp + pix) * C;
    float* lp = dst_lo ? dst_lo + ((size_t)b * Hp * Wp + pix) * C : nullptr;
    if (!inside) {
      for (int c = 0; c < C; ++c) {
        dp[c] = 0.f;
        if (lp) lp[c] = 0.f;
      }
      continue;
    }
    const float* sp = src + (size_t)b * Cs * plane + (size_t)y * W + x;
    if (mode == 0) {
      for (int c = 0; c < C; ++c) {
        const float v = c < Cs ? __ldg(sp + c * plane) : 0.f;
        if (lp) {
          const float h = tf32_rna(v);
          dp[c] = h, lp[c] = tf32_rna(v - h);
        } else {
          dp[c] = v;
        }
      }
    } else {
      float3 rgb;
      if (mode == 1) {
        rgb = make_float3(__ldg(sp), __ldg(sp + plane), __ldg(sp + 2 * plane));
      } else if (mode == 2) {
        const float g = (__ldg(sp) * 1.0f + 50.0f) / 100.0f;  // util.py:63,97-101
        rgb = make_float3(g, g, g);
      } else {
        rgb = lab_to_srgb(__ldg(sp) + 50.0f, __ldg(sp + plane), __ldg(sp + 2 * plane));
      }
      // util.py:347-352: BGR order, minus mean, times 255
      dp[0] = (rgb.z - 0.40760392f) * 255.f;
      dp[1] = (rgb.y - 0.45795686f) * 255.f;
      dp[2] = (rgb.x - 0.48501961f) * 255.f;
      for (int c = 3; c < C; ++c) dp[c] = 0.f;
    }
  }
}

// interior of a padded NHWC activation -> NCHW.  One block = 32 pixels x 32 channels via smem transpose.
__global__ void __launch_bounds__(256) act_to_nchw_kernel(const float* __restrict__ src, const float* __restrict__ src_lo,
                                                          int H, int W, int P, int sC, int sCoff, int C,
                                                          float* __restrict__ dst) {
  __shared__ float t[32][33];
  const int b = blockIdx.z;
  const int Hp = H + 2 * P, Wp = W + 2 * P;
  const int pix0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 8 rows per pass
  for (int r = ty; r < 32; r += 8) {
    const int pix = pix0 + r;
    float v = 0.f;
    if (pix < H * W && c0 + tx < C) {
      const int y = pix / W, x = pix - y * W;
      const size_t o = (((size_t)b * Hp + y + P) * Wp + x + P) * sC + sCoff + c0 + tx;
      v = __ldg(src + o);
      if (src_lo) v += __ldg(src_lo + o);
    }
    t[r][tx] = v;
  }
  __syncthreads();
  for (int r = ty; r < 32; r += 8) {
    const int c = c0 + r, pix = pix0 + tx;
    if (c < C && pix < H * W) dst[((size_t)b * C + c) * H * W + pix] = t[tx][r];
  }
}

__global__ void __launch_bounds__(256) maxpool2_kernel(const float* __restrict__ src, const float* __restrict__ src_lo,
                                                       int sH, int sW, int sP, int C, float* __restrict__ dst,
                                                       float* __restrict__ dst_lo, int dP) {
  const int b = blockIdx.y;
  const int dH = sH / 2, dW = sW / 2;
  const int dHp = dH + 2 * dP, dWp = dW + 2 * dP, sHp = sH + 2 * sP, sWp = sW + 2 * sP;
  const int c4n = C >> 2;
  const long total = (long)dHp * dWp * c4n;
  for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
    const int c = (int)(idx % c4n) * 4;
    const int pix = (int)(idx / c4n);
    const int yp = pix / dWp, xp = pix - yp * dWp;
    const int y = yp - dP, x = xp - dP;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (y >= 0 && y < dH && x >= 0 && x < dW) {
      const size_t so = (((size_t)b * sHp + 2 * y + sP) * sWp + 2 * x + sP) * C + c;
      const float4 a = ld4(src, src_lo, so);
      const float4 b4 = ld4(src, src_lo, so + C);
      const float4 c4 = ld4(src, src_lo, so + (size_t)sWp * C);
      const float4 d = ld4(src, src_lo, so + (size_t)sWp * C + C);
      v.x = fmaxf(fmaxf(a.x, b4.x), fmaxf(c4.x, d.x));
      v.y = fmaxf(fmaxf(a.y, b4.y), fmaxf(c4.y, d.y));
      v.z = fmaxf(fmaxf(a.z, b4.z), fmaxf(c4.z, d.z));
      v.w = fmaxf(fmaxf(a.w, b4.w), fmaxf(c4.w, d.w));
    }
    st4(dst, dst_lo, ((size_t)b * dHp * dWp + pix) * C + c, v);
  }
}

// the two kernels above for fp16 hi/lo planes with a device-side exponent
__global__ void __launch_bounds__(256) act_to_nchw_h16_kernel(const __half* __restrict__ hp, const __half* __restrict__ lp,
                                                              const ScaleCell* __restrict__ cell, int H, int W, int P, int sC,
                                                              int C, float* __restrict__ dst) {
  __shared__ float t[32][33];
  const float descale = exp2_int(-cell->e);
  const int b = blockIdx.z;
  const int Hp = H + 2 * P, Wp = W + 2 * P;
  const int pix0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int r = ty; r < 32; r += 8) {
    const int pix = pix0 + r;
    float v = 0.f;
    if (pix < H * W && c0 + tx < C) {
      const int y = pix / W, x = pix - y * W;
      const size_t o = (((size_t)b * Hp + y + P) * Wp + x + P) * sC + c0 + tx;
      v = (__half2float(hp[o]) + __half2float(lp[o])) * descale;
    }
    t[r][tx] = v;
  }
  __syncthreads();
  for (int r = ty; r < 32; r += 8) {
    const int c = c0 + r, pix = pix0 + tx;
    if (c < C && pix < H * W) dst[((size_t)b * C + c) * H * W + pix] = t[tx][r];
  }
}

__global__ void __launch_bounds__(256) maxpool2_h16_kernel(const __half* __restrict__ hp, const __half* __restrict__ lp,
                                                           const ScaleCell* __restrict__ cell_in, int sH, int sW, int sP, int C,
                                                           __half* __restrict__ dh, __half* __restrict__ dl,
                                                           ScaleCell* __restrict__ cell_out, int dP) {
  const int b = blockIdx.y;
  if (b == 0 && blockIdx.x == 0 && threadIdx.x == 0) *cell_out = *cell_in;  // same scale, same max (values are >= 0)
  const int dH = sH / 2, dW = sW / 2;
  const int dHp = dH + 2 * dP, dWp = dW + 2 * dP, sHp = sH + 2 * sP, sWp = sW + 2 * sP;
  const int c4n = C >> 2;
  const long total = (long)dHp * dWp * c4n;
  for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
    const int c = (int)(idx % c4n) * 4;
    const int pix = (int)(idx / c4n);
    const int yp = pix / dWp, xp = pix - yp * dWp;
    const int y = yp - dP, x = xp - dP;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (y >= 0 && y < dH && x >= 0 && x < dW) {
      const size_t so = (((size_t)b * sHp + 2 * y + sP) * sWp + 2 * x + sP) * C + c;
      const float4 a = ld4h(hp, lp, so);
      const float4 b4 = ld4h(hp, lp, so + C);
      const float4 c4 = ld4h(hp, lp, so + (size_t)sWp * C);
      const float4 d = ld4h(hp, lp, so + (size_t)sWp * C + C);
      v.x = fmaxf(fmaxf(a.x, b4.x), fmaxf(c4.x, d.x));
      v.y = fmaxf(fmaxf(a.y, b4.y), fmaxf(c4.y, d.y));
      v.z = fmaxf(fmaxf(a.z, b4.z), fmaxf(c4.z, d.z));
      v.w = fmaxf(fmaxf(a.w, b4.w), fmaxf(c4.w, d.w));
    }
    st4h(dh, dl, ((size_t)b * dHp * dWp + pix) * C + c, v, 1.f);  // re-splitting hi + lo is exact
  }
}

__global__ void __launch_bounds__(256) amax_kernel(const float4* __restrict__ x, size_t n4, ScaleCell* __restrict__ cell) {
  __shared__ float red[8];
  float m = 0.f;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
    const float4 v = __ldg(x + i);
    m = fmaxf(fmaxf(m, fmaxf(fabsf(v.x), fabsf(v.y))), fmaxf(fabsf(v.z), fabsf(v.w)));
  }
  block_amax_commit(m, cell, red);
}

__global__ void __launch_bounds__(256) avgpool4_lab_kernel(const float* __restrict__ src, float* __restrict__ V, int H,
                                                           int W) {
  const int b = blockIdx.y;
  const int h = H / 4, w = W / 4;
  for (int n = blockIdx.x * blockDim.x + threadIdx.x; n < h * w; n += gridDim.x * blockDim.x) {
    const int i = n / w, j = n - i * w;
    float o[3];
    for (int c = 0; c < 3; ++c) {
      const float* sp = src + ((size_t)b * 3 + c) * H * W + (size_t)(4 * i) * W + 4 * j;
      float s = 0.f;
      for (int dy = 0; dy < 4; ++dy)
        for (int dx = 0; dx < 4; ++dx) s += __ldg(sp + dy * W + dx);
      o[c] = s * (1.0f / 16.0f);
    }
    // 4th lane = 1: the softmax epilogue of the correlation accumulates (b, sum of weights) with one packed FMA
    *reinterpret_cast<float4*>(V + ((size_t)b * h * w + n) * 4) = make_float4(o[0], o[1], o[2], 1.f);
  }
}

__global__ void __launch_bounds__(256) pack_v4_kernel(const float* __restrict__ src3, float* __restrict__ dst4, size_t n) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    if (src3)
      reinterpret_cast<float4*>(dst4)[i] = make_float4(__ldg(src3 + 3 * i), __ldg(src3 + 3 * i + 1), __ldg(src3 + 3 * i + 2), 1.f);
    else
      dst4[4 * i + 3] = 1.f;
  }
}

__global__ void __launch_bounds__(256) rows_to_nchw_up4_kernel(const float* __restrict__ yrows,
                                                               const float* __restrict__ simrows, float* __restrict__ y,
                                                               float* __restrict__ sim, int h, int w) {
  const int b = blockIdx.y;
  const int H = 4 * h, W = 4 * w;
  for (int pix = blockIdx.x * blockDim.x + threadIdx.x; pix < H * W; pix += gridDim.x * blockDim.x) {
    const int i = pix / W, j = pix - i * W;
    const int n = (i >> 2) * w + (j >> 2);
    const float4 v = __ldg(reinterpret_cast<const float4*>(yrows + ((size_t)b * h * w + n) * 4));
    if (y) {
      y[((size_t)b * 3 + 0) * H * W + pix] = v.x;
      y[((size_t)b * 3 + 1) * H * W + pix] = v.y;
      y[((size_t)b * 3 + 2) * H * W + pix] = v.z;
    }
    if (sim) sim[(size_t)b * H * W + pix] = __ldg(simrows + (size_t)b * h * w + n);
  }
}

__global__ void __launch_bounds__(256) build_color_input_kernel(const float* __restrict__ IA_l,
                                                                const float* __restrict__ yrows,
                                                                const float* __restrict__ simrows,
                                                                const float* __restrict__ last, float* __restrict__ dst,
                                                                int H, int W, int P) {
  const int b = blockIdx.y;
  const int Hp = H + 2 * P, Wp = W + 2 * P;
  const int h = H / 4, w = W / 4;
  const size_t plane = (size_t)H * W;
  for (int pix = blockIdx.x * blockDim.x + threadIdx.x; pix < Hp * Wp; pix += gridDim.x * blockDim.x) {
    const int yp = pix / Wp, xp = pix - yp * Wp;
    const int y = yp - P, x = xp - P;
    float4 o0 = make_float4(0.f, 0.f, 0.f, 0.f), o1 = o0;
    if (y >= 0 && y < H && x >= 0 && x < W) {
      const size_t q = (size_t)y * W + x;
      const int n = (y >> 2) * w + (x >> 2);
      const float4 yr = __ldg(reinterpret_cast<const float4*>(yrows + ((size_t)b * h * w + n) * 4));
      o0.x = __ldg(IA_l + (size_t)b * plane + q);
      o0.y = yr.y;  // warped a (channel 1 of the warped Lab, FrameColor.py:63)
      o0.z = yr.z;  // warped b
      o0.w = __ldg(simrows + (size_t)b * h * w + n);
      o1.x = __ldg(last + ((size_t)b * 3 + 0) * plane + q);
      o1.y = __ldg(last + ((size_t)b * 3 + 1) * plane + q);
      o1.z = __ldg(last + ((size_t)b * 3 + 2) * plane + q);
    }
    float4* dp = reinterpret_cast<float4*>(dst + ((size_t)b * Hp * Wp + pix) * 8);
    dp[0] = o0;
    dp[1] = o1;
  }
}

// warp per pixel: 1x1 conv C -> 2, tanh * 128
__global__ void __launch_bounds__(256) final_ab_kernel(const float* __restrict__ x, int H, int W, int P, int C,
                                                       const float* __restrict__ w, const float* __restrict__ bias,
                                                       float* __restrict__ out) {
  const int b = blockIdx.y;
  const int lane = threadIdx.x & 31;
  const int Hp = H + 2 * P, Wp = W + 2 * P;
  const int warps = gridDim.x * (blockDim.x >> 5);
  const int nv = C / 128;  // float4 per lane (C = 128 -> 1)
  for (int pix = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); pix < H * W; pix += warps) {
    const int y = pix / W, xx = pix - y * W;
    const float* sp = x + (((size_t)b * Hp + y + P) * Wp + xx + P) * C;
    float s0 = 0.f, s1 = 0.f;
    for (int i = 0; i < nv; ++i) {
      const int c = (i * 32 + lane) * 4;
      const float4 v = __ldg(reinterpret_cast<const float4*>(sp + c));
      const float4 w0 = __ldg(reinterpret_cast<const float4*>(w + c));
      const float4 w1 = __ldg(reinterpret_cast<const float4*>(w + C + c));
      s0 += v.x * w0.x + v.y * w0.y + v.z * w0.z + v.w * w0.w;
      s1 += v.x * w1.x + v.y * w1.y + v.z * w1.z + v.w * w1.w;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      s0 += __shfl_xor_sync(0xffffffffu, s0, o);
      s1 += __shfl_xor_sync(0xffffffffu, s1, o);
    }
    if (lane == 0) {
      out[((size_t)b * 2 + 0) * H * W + pix] = tanhf(s0 + bias[0]) * 128.f;
      out[((size_t)b * 2 + 1) * H * W + pix] = tanhf(s1 + bias[1]) * 128.f;
    }
  }
}

__global__ void __launch_bounds__(256) make_last_kernel(const float* __restrict__ IA_l, const float* __restrict__ ab,
                                                        float* __restrict__ last, int HW) {
  const int b = blockIdx.y;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < HW; i += gridDim.x * blockDim.x) {
    last[((size_t)b * 3 + 0) * HW + i] = IA_l[(size_t)b * HW + i];
    last[((size_t)b * 3 + 1) * HW + i] = ab[((size_t)b * 2 + 0) * HW + i];
    last[((size_t)b * 3 + 2) * HW + i] = ab[((size_t)b * 2 + 1) * HW + i];
  }
}

__global__ void __launch_bounds__(256) transpose_cn_kernel(const float* __restrict__ src, float* __restrict__ dst, int R,
                                                           int Cc) {
  // src [b][R][Cc] -> dst [b][Cc][R]
  __shared__ float t[32][33];
  const int b = blockIdx.z;
  const int r0 = blockIdx.y * 32, c0 = blockIdx.x * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int r = ty; r < 32; r += 8)
    t[r][tx] = (r0 + r < R && c0 + tx < Cc) ? src[((size_t)b * R + r0 + r) * Cc + c0 + tx] : 0.f;
  __syncthreads();
  for (int r = ty; r < 32; r += 8)
    if (c0 + r < Cc && r0 + tx < R) dst[((size_t)b * Cc + c0 + r) * R + r0 + tx] = t[tx][r];
}

// F.interpolate(x, scale_factor=0.5, mode="bilinear") (test.py:58,71) for even sizes: the sample point of output
// (i, j) is source (2i + 0.5, 2j + 0.5), i.e. the mean of a 2x2 block with weights 0.5 * 0.5.
__global__ void __launch_bounds__(256) resize_half_kernel(const float* __restrict__ src, float* __restrict__ dst, int planes,
                                                          int H, int W) {
  const int h = H / 2, w = W / 2;
  const long total = (long)planes * h * w;
  for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
    const int j = (int)(idx % w);
    const long t = idx / w;
    const int i = (int)(t % h);
    const long pl = t / h;
    const float* sp = src + (pl * H + 2 * i) * W + 2 * j;
    const float2 a = __ldg(reinterpret_cast<const float2*>(sp)), b = __ldg(reinterpret_cast<const float2*>(sp + W));
    // torch: lambda = 0.5 on both axes: (a0*0.5 + a1*0.5) * 0.5 + (b0*0.5 + b1*0.5) * 0.5, rows first
    dst[idx] = 0.5f * (0.5f * a.x + 0.5f * a.y) + 0.5f * (0.5f * b.x + 0.5f * b.y);
  }
}

// F.interpolate(x, scale_factor=2, mode="bilinear") * scale (test.py:100-102, align_corners=False): output I samples
// source I/2 - 0.25, clamped at the borders -> weights (0.25, 0.75) / (0.75, 0.25) on neighbouring source pixels.
__global__ void __launch_bounds__(256) upsample2_kernel(const float* __restrict__ src, float* __restrict__ dst, int planes,
                                                        int h, int w, float scale) {
  const int H = 2 * h, W = 2 * w;
  const long total = (long)planes * H * W;
  for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
    const int J = (int)(idx % W);
    const long t = idx / W;
    const int I = (int)(t % H);
    const long pl = t / H;
    // source index and weight like torch's area_pixel_compute_source_index (negative coordinates clamp to 0)
    float sy = (I + 0.5f) * 0.5f - 0.5f, sx = (J + 0.5f) * 0.5f - 0.5f;
    sy = sy < 0.f ? 0.f : sy, sx = sx < 0.f ? 0.f : sx;
    const int y0 = (int)sy, x0 = (int)sx;
    const int y1 = y0 + (y0 < h - 1 ? 1 : 0), x1 = x0 + (x0 < w - 1 ? 1 : 0);
    const float ly = sy - y0, lx = sx - x0;
    const float* sp = src + pl * h * w;
    const float v00 = __ldg(sp + (long)y0 * w + x0), v01 = __ldg(sp + (long)y0 * w + x1);
    const float v10 = __ldg(sp + (long)y1 * w + x0), v11 = __ldg(sp + (long)y1 * w + x1);
    const float v = (1.f - ly) * ((1.f - lx) * v00 + lx * v01) + ly * ((1.f - lx) * v10 + lx * v11);
    dst[idx] = v * scale;
  }
}

inline int grid_for(long total, int threads, int cap = 148 * 16) {
  long g = (total + threads - 1) / threads;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return (int)g;
}

}  // namespace

void launch_xform(const XformParams& p, int B, cudaStream_t s) {
  const long total = (long)(p.dH + 2 * p.dP) * (p.dW + 2 * p.dP) * (p.C / 8);
  dim3 grid(grid_for(total, 256), B);
  const size_t sm = p.stats ? 2 * p.C * sizeof(float) : 0;
  xform_kernel<<<grid, 256, sm, s>>>(p);
  launch_counter_add(1);
}

void launch_pixnorm(const PixNormParams& p, int B, cudaStream_t s) {
  const long pix = (long)(p.sH + 2 * p.dP) * (p.sW + 2 * p.dP);
  dim3 grid(grid_for(pix, 8), B);
  switch (p.C) {
    case 128: pixnorm_kernel<1><<<grid, 256, 0, s>>>(p); break;
    case 256: pixnorm_kernel<2><<<grid, 256, 0, s>>>(p); break;
    case 512: pixnorm_kernel<4><<<grid, 256, 0, s>>>(p); break;
    default: break;  // validated by the caller
  }
  launch_counter_add(1);
}

void launch_nchw_to_act(const float* src, int Cs, float* dst, float* dst_lo, int B, int H, int W, int C, int P,
                        int pad_mode, int mode, cudaStream_t s) {
  dim3 grid(grid_for((long)(H + 2 * P) * (W + 2 * P), 256), B);
  nchw_to_act_kernel<<<grid, 256, 0, s>>>(src, Cs, dst, dst_lo, H, W, C, P, pad_mode, mode);
  launch_counter_add(1);
}

void launch_act_to_nchw(const float* src, const float* src_lo, int H, int W, int P, int sC, int sCoff, int C, float* dst,
                        int B, cudaStream_t s) {
  dim3 grid((H * W + 31) / 32, (C + 31) / 32, B);
  act_to_nchw_kernel<<<grid, 256, 0, s>>>(src, src_lo, H, W, P, sC, sCoff, C, dst);
  launch_counter_add(1);
}

void launch_maxpool2(const float* src, const float* src_lo, int sH, int sW, int sP, int C, float* dst, float* dst_lo,
                     int dP, int B, cudaStream_t s) {
  const long total = (long)(sH / 2 + 2 * dP) * (sW / 2 + 2 * dP) * (C / 4);
  dim3 grid(grid_for(total, 256), B);
  maxpool2_kernel<<<grid, 256, 0, s>>>(src, src_lo, sH, sW, sP, C, dst, dst_lo, dP);
  launch_counter_add(1);
}

void launch_act_to_nchw_h16(const void* h16, const void* l16, const ScaleCell* cell, int H, int W, int P, int sC, int C,
                            float* dst, int B, cudaStream_t s) {
  dim3 grid((H * W + 31) / 32, (C + 31) / 32, B);
  act_to_nchw_h16_kernel<<<grid, 256, 0, s>>>(reinterpret_cast<const __half*>(h16), reinterpret_cast<const __half*>(l16), cell, H, W,
                                              P, sC, C, dst);
  launch_counter_add(1);
}

void launch_maxpool2_h16(const void* h16, const void* l16, const ScaleCell* cell_in, int sH, int sW, int sP, int C, void* dh16,
                         void* dl16, ScaleCell* cell_out, int dP, int B, cudaStream_t s) {
  const long total = (long)(sH / 2 + 2 * dP) * (sW / 2 + 2 * dP) * (C / 4);
  dim3 grid(grid_for(total, 256), B);
  maxpool2_h16_kernel<<<grid, 256, 0, s>>>(reinterpret_cast<const __half*>(h16), reinterpret_cast<const __half*>(l16), cell_in, sH, sW,
                                           sP, C, reinterpret_cast<__half*>(dh16), reinterpret_cast<__half*>(dl16), cell_out, dP);
  launch_counter_add(1);
}

void launch_amax(const float* x, size_t n, ScaleCell* cell, cudaStream_t s) {
  amax_kernel<<<(unsigned)grid_for((long)(n / 4), 256, 148 * 4), 256, 0, s>>>(reinterpret_cast<const float4*>(x), n / 4, cell);
  launch_counter_add(1);
}

void launch_avgpool4_lab(const float* src, float* V, int B, int H, int W, cudaStream_t s) {
  dim3 grid(grid_for((long)(H / 4) * (W / 4), 256), B);
  avgpool4_lab_kernel<<<grid, 256, 0, s>>>(src, V, H, W);
  launch_counter_add(1);
}

void launch_pack_v4(const float* src3, float* dst4, size_t n, cudaStream_t s) {
  pack_v4_kernel<<<grid_for((long)n, 256), 256, 0, s>>>(src3, dst4, n);
  launch_counter_add(1);
}

void launch_rows_to_nchw_up4(const float* yrows, const float* simrows, float* y, float* sim, int B, int h, int w,
                             cudaStream_t s) {
  dim3 grid(grid_for((long)16 * h * w, 256), B);
  rows_to_nchw_up4_kernel<<<grid, 256, 0, s>>>(yrows, simrows, y, sim, h, w);
  launch_counter_add(1);
}

void launch_build_color_input(const float* IA_l, const float* yrows, const float* simrows, const float* last_lab,
                              float* dst, int B, int H, int W, int P, cudaStream_t s) {
  dim3 grid(grid_for((long)(H + 2 * P) * (W + 2 * P), 256), B);
  build_color_input_kernel<<<grid, 256, 0, s>>>(IA_l, yrows, simrows, last_lab, dst, H, W, P);
  launch_counter_add(1);
}

void launch_final_ab(const float* x, int H, int W, int P, int C, const float* w, const float* bias, float* out, int B,
                     cudaStream_t s) {
  dim3 grid(grid_for((long)H * W, 8), B);
  final_ab_kernel<<<grid, 256, 0, s>>>(x, H, W, P, C, w, bias, out);
  launch_counter_add(1);
}

void launch_make_last(const float* IA_l, const float* ab, float* last, int B, int H, int W, cudaStream_t s) {
  dim3 grid(grid_for((long)H * W, 256), B);
  make_last_kernel<<<grid, 256, 0, s>>>(IA_l, ab, last, H * W);
  launch_counter_add(1);
}

namespace {
struct Mat3 {
  double m[9];
};
// util.py:134-151 -> skimage.color.lab2rgb, all in float64 like the reference; one thread per pixel
__global__ void __launch_bounds__(256) lab_to_rgb8_kernel(const float* __restrict__ l, const float* __restrict__ ab,
                                                          unsigned char* __restrict__ rgb, int HW, const Mat3 M) {
  const int b = blockIdx.y;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < HW; i += gridDim.x * blockDim.x) {
    const double L = (double)l[(size_t)b * HW + i] + 50.0;  // l_norm = 1, l_mean = 50 (util.py:15-18)
    const double A = (double)ab[((size_t)b * 2 + 0) * HW + i], Bq = (double)ab[((size_t)b * 2 + 1) * HW + i];
    double f[3];
    f[1] = (L + 16.0) / 116.0;
    f[0] = A / 500.0 + f[1];
    f[2] = f[1] - Bq / 200.0;
    if (f[2] < 0.0) f[2] = 0.0;
    const double white[3] = {0.95047, 1.0, 1.08883};
    double xyz[3];
#pragma unroll
    for (int k = 0; k < 3; ++k)
      xyz[k] = (f[k] > 0.2068966 ? f[k] * f[k] * f[k] : (f[k] - 16.0 / 116.0) / 7.787) * white[k];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      double v = xyz[0] * M.m[k * 3 + 0] + xyz[1] * M.m[k * 3 + 1] + xyz[2] * M.m[k * 3 + 2];
      v = v > 0.0031308 ? 1.055 * pow(v, 1.0 / 2.4) - 0.055 : v * 12.92;
      v = fmin(fmax(v, 0.0), 1.0);
      rgb[((size_t)b * HW + i) * 3 + k] = (unsigned char)(v * 255.0);
    }
  }
}
}  // namespace

namespace {
// util_distortion.py:18-23 -> skimage.color.rgb2lab in float64, then ToTensor (.float()) and Normalize (L - 50)
__global__ void __launch_bounds__(256) rgb8_to_lab_kernel(const unsigned char* __restrict__ rgb, float* __restrict__ lab, int HW) {
  const int b = blockIdx.y;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < HW; i += gridDim.x * blockDim.x) {
    const unsigned char px[3] = {rgb[((size_t)b * HW + i) * 3 + 0], rgb[((size_t)b * HW + i) * 3 + 1], rgb[((size_t)b * HW + i) * 3 + 2]};
    float L, A, Bq;
    rgb8_to_lab_px(px, &L, &A, &Bq);
    lab[((size_t)b * 3 + 0) * HW + i] = L;
    lab[((size_t)b * 3 + 1) * HW + i] = A;
    lab[((size_t)b * 3 + 2) * HW + i] = Bq;
  }
}
}  // namespace

void launch_rgb8_to_lab(const unsigned char* rgb, float* lab, int B, int H, int W, cudaStream_t s) {
  dim3 grid(grid_for((long)H * W, 256), B);
  rgb8_to_lab_kernel<<<grid, 256, 0, s>>>(rgb, lab, H * W);
  launch_counter_add(1);
}

void launch_lab_to_rgb8(const float* l, const float* ab, unsigned char* rgb, int B, int H, int W, const double* rgb_from_xyz,
                        cudaStream_t s) {
  Mat3 M;
  for (int i = 0; i < 9; ++i) M.m[i] = rgb_from_xyz[i];
  dim3 grid(grid_for((long)H * W, 256), B);
  lab_to_rgb8_kernel<<<grid, 256, 0, s>>>(l, ab, rgb, H * W, M);
  launch_counter_add(1);
}

void launch_resize_half(const float* src, float* dst, int planes, int H, int W, cudaStream_t s) {
  resize_half_kernel<<<grid_for((long)planes * (H / 2) * (W / 2), 256), 256, 0, s>>>(src, dst, planes, H, W);
  launch_counter_add(1);
}

void launch_upsample2(const float* src, float* dst, int planes, int h, int w, float scale, cudaStream_t s) {
  upsample2_kernel<<<grid_for((long)planes * 4 * h * w, 256), 256, 0, s>>>(src, dst, planes, h, w, scale);
  launch_counter_add(1);
}

void launch_transpose_cn(const float* src, float* dst, int B, int R, int Cc, cudaStream_t s) {
  // src [B][R][Cc] -> dst [B][Cc][R]
  dim3 grid((Cc + 31) / 32, (R + 31) / 32, B);
  transpose_cn_kernel<<<grid, 256, 0, s>>>(src, dst, R, Cc);
  launch_counter_add(1);
}

}  // namespace dvc
