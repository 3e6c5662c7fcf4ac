// libdvc.so host side: context, weight packing, the three layer programs (VGG19 trunk, WarpNet,
// ColorVidNet) expressed over the kernels of this directory, and the C ABI of include/dvc.h.
//
// Reference interfaces replaced (file:line in the reference tree):
//   VGG19_pytorch.forward   models/NonlocalNet.py:228-256
//   WarpNet.forward         models/NonlocalNet.py:427-502
//   ColorVidNet.forward     models/ColorVidNet.py:96-144
//   frame_colorization      models/FrameColor.py:41-67, per-clip loop test.py:57-96
#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <functional>
#include <map>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/dvc.h"
#include "conv_tc.cuh"
#include "corr_tc.cuh"
#include "dvc_internal.cuh"

namespace dvc {

static std::atomic<int64_t> g_launches{0};
int64_t launch_counter_add(int64_t n) { return g_launches.fetch_add(n) + n; }

struct ConvW {
  float* w = nullptr;  // [taps][cin_pad][cout_pad]       (CUDA-core kernel: output channels contiguous)
  float* b = nullptr;  // [cout_pad]
  float* wt_hi = nullptr;  // [taps][cout_pad_tc][cin_pad]  tf32 hi plane (tensor-core kernel: K contiguous)
  float* wt_lo = nullptr;  //                               tf32 lo plane
  void* w16_hi = nullptr;  // [taps][cout_pad_tc][cin_pad]  fp16 hi plane of w * 2^e_w
  void* w16_lo = nullptr;
  int e_w = 0;
  float l1max = 0.f;  // max over output channels of sum |w| (bounds |conv output| by l1max * max|input| + bmax)
  float bmax = 0.f;   // max |bias|
  int cin = 0, cin_pad = 0, cout = 0, cout_pad = 0, cout_pad_tc = 0, k = 0;
};

// exponent e such that |x| <= bound implies |x * 2^e| <= 2^15 (fp16 max 65504), clamped to a sane range
static inline int e16_for(double bound) {
  if (!(bound > 0)) return 14;
  int e = (int)floor(log2(32768.0 / bound));
  return e > 14 ? 14 : (e < -14 ? -14 : e);
}
static inline unsigned short host_f2h(float f) {  // fp32 -> fp16 bits, round to nearest even, subnormals kept
  uint32_t x;
  memcpy(&x, &f, 4);
  const uint32_t sign = (x >> 16) & 0x8000u;
  const int32_t exp = (int32_t)((x >> 23) & 0xff) - 127 + 15;
  uint32_t man = x & 0x7fffffu;
  if (((x >> 23) & 0xff) == 0xff) return (unsigned short)(sign | 0x7c00u | (man ? 0x200u : 0));
  if (exp >= 31) return (unsigned short)(sign | 0x7bffu);  // saturate instead of inf
  if (exp <= 0) {
    if (exp < -10) return (unsigned short)sign;
    man |= 0x800000u;
    const int shift = 14 - exp;
    uint32_t h = man >> shift;
    const uint32_t rem = man & ((1u << shift) - 1), half = 1u << (shift - 1);
    if (rem > half || (rem == half && (h & 1))) h++;
    return (unsigned short)(sign | h);
  }
  uint32_t h = ((uint32_t)exp << 10) | (man >> 13);
  const uint32_t rem = man & 0x1fffu;
  if (rem > 0x1000u || (rem == 0x1000u && (h & 1))) h++;
  return (unsigned short)(sign | h);
}
static inline float host_h2f(unsigned short h) {
  const uint32_t sign = (uint32_t)(h & 0x8000u) << 16;
  const uint32_t exp = (h >> 10) & 0x1f, man = h & 0x3ffu;
  float f;
  if (exp == 0) {
    f = ldexpf((float)man, -24);
  } else if (exp == 31) {
    f = man ? NAN : INFINITY;
  } else {
    f = ldexpf((float)(man | 0x400u), (int)exp - 25);
  }
  uint32_t u;
  memcpy(&u, &f, 4);
  u |= sign;
  memcpy(&f, &u, 4);
  return f;
}
// fp16 hi/lo planes of v * 2^e: returns device buffers
static void host_split16(const std::vector<float>& v, int e, std::vector<unsigned short>& hi, std::vector<unsigned short>& lo) {
  hi.resize(v.size()), lo.resize(v.size());
  for (size_t i = 0; i < v.size(); ++i) {
    const float x = ldexpf(v[i], e);
    hi[i] = host_f2h(x);
    lo[i] = host_f2h(x - host_h2f(hi[i]));
  }
}

static inline float host_tf32_rna(float x) {  // cvt.rna.tf32.f32: nearest, ties away, 10 explicit mantissa bits
  uint32_t u;
  memcpy(&u, &x, 4);
  if ((u & 0x7f800000u) == 0x7f800000u) return x;
  u = (u + 0x1000u) & 0xffffe000u;
  float r;
  memcpy(&r, &u, 4);
  return r;
}

struct Buf {
  void* p = nullptr;
  size_t bytes = 0;
  int sig[5] = {0, 0, 0, 0, 0};
};

}  // namespace dvc

using namespace dvc;

struct dvc_ctx {
  int device = 0;
  std::string err;
  std::unordered_map<std::string, ConvW> conv[3];
  std::unordered_map<std::string, float> slope[3];
  std::unordered_map<std::string, float*> vec[3];
  std::unordered_map<std::string, std::vector<float>> host_bias[3];  // bias seen before its weight
  int num_sms = 148;
  // default: tensor cores with fp32-class accuracy (3xTF32); DVC_MATH_FP32 selects the exact CUDA-core engines
  int conv_math = DVC_MATH_TF32X3, corr_math = DVC_MATH_FP16X3;
  int tc_kbytes = 128;    // tensor-core convolutions: K bytes per pipeline stage (64 or 128, see conv_tc.cu)
  CorrPeers corr_peers;   // fused all-gather targets of dvc_corr_softmax_warp (dvc_corr_set_peer_outputs)
  ScaleCell* cell_next = nullptr;
  int cell_left = 0;
  int corr_cluster = 2;   // correlation: 2 = CTA pairs (tcgen05.mma.cta_group::2), 1 = single CTAs
  // stand-alone correlation entry: the caller promises that the phi_hat / V buffers keep their contents while this is set, so
  // their transposed / packed / split forms are prepared once per (pointer, size) -- the exemplar side of a clip
  int corr_phi_static = 0;
  const void* corr_phi_key = nullptr;
  const void* corr_V_key = nullptr;
  long long corr_phi_dims = 0, corr_phi_version = 0;
  int corr_screen = 1;    // T <= 2e-10, FP16X3: one screening pass + exact re-scoring of the candidates (0: exact 3-pass kernel)
  CorrWorkspace corr_ws;  // operand planes + split partials of the tensor-core correlation (pre-sized by dvc_set_exemplar)
  CorrWorkspace corr_ws2;  // the same for the second phase-A stream of the clip driver (clip_astreams = 2)
  int clip_astreams = 1;   // clip driver: 1 = frame t+1's phase A overlaps frame t's ColorVidNet; 2 = frames t+1 AND t+2
  long long ex_version = 0;  // bumped whenever ex_phi's contents change (the correlation caches the exemplar's planes)
  int tc_dbg = 0;         // timing experiments of the conv engine (wrong results): see ConvTcParams::dbg
  int tc_rowshare = 0;    // tensor-core convolutions: taps of a kernel row share one activation tile (conv_tc.cu: CfgRS)
  int tc_force_bn = 0;    // tests: channel tile (64 / 128 / 256) forced on every tensor-core convolution it divides
  int tc_tail = 0;        // tensor-core convolutions: 1 = 128-channel tiles for the partial last round of 256-channel
                          // launches (-1.3 % on one stream, +1.6 % in the two-stream clip pipeline: off by default)
  int tc_f16 = 1;         // tensor-core convolutions: fp16 hi/lo planes for layers with provably bounded inputs
  std::unordered_map<std::string, float> vec_absmax[3];  // max |scale| of the *_ss vectors
  int tc_cluster = 2;     // tensor-core convolutions: 2 = CTA pairs (tcgen05.mma.cta_group::2), 1 = single CTAs
  int tc_kc = 1;          // tensor-core convolutions: k-blocks per TMEM chunk (see conv_tc.cu)
  bool two_level = true;  // fp32 convolutions: per-tap two-level accumulation (see conv_simt.cu)
  std::map<std::string, Buf> bufs;
  // InstanceNorm statistics arena (doubles), bump-allocated per forward call
  double* stats = nullptr;
  size_t stats_cap = 0, stats_used = 0, stats_lo = 0, stats_hi = 0;
  int cur_arena = 0;          // 0: frame-independent phase, 1: ColorVidNet (may run concurrently on two streams)
  int tc_epoch[3] = {0, 0, 0};   // split-K hand-over epochs, one flag buffer per arena
  int tc_splits = 1;          // split-K: 1 = off (default: measured no gain once two streams overlap), 0 = automatic, >1 = forced
  // clip driver: frame t+1's VGG/WarpNet/correlation overlaps frame t's ColorVidNet on two internal streams
  cudaStream_t sA = nullptr, sC = nullptr, sU = nullptr, sD = nullptr;  // phase A, phase C, uploads, downloads
  cudaStream_t sA2 = nullptr;  // phase A of the odd frames when clip_astreams = 2
  cudaEvent_t evJoinA2 = nullptr;
  cudaEvent_t evA[4] = {nullptr, nullptr, nullptr, nullptr}, evC[4] = {nullptr, nullptr, nullptr, nullptr}, evFork = nullptr,
              evJoinA = nullptr, evJoinC = nullptr, evJoinD = nullptr;
  cudaEvent_t evU[4] = {nullptr, nullptr, nullptr, nullptr}, evD[4] = {nullptr, nullptr, nullptr, nullptr};
  // video driver (dvc_colorize_video_rgb8): post-processing + download stream, one event per batch slot of the rings
  cudaStream_t sP = nullptr;
  cudaEvent_t evP[2] = {nullptr, nullptr}, evJoinP = nullptr;
  int video_batch = 8;  // frames per dvc_postprocess_rgb8 batch in the video driver (DESIGN.md §4.5: measured)
  // recurrence state of dvc_colorize_video_rgb8 ("vid.last"): valid for this exemplar version and output size only
  long long vid_ex_version = -1;
  int vid_Ho = 0, vid_Wo = 0;
  // exemplar cache
  float* ex_phi = nullptr;  // [N][256]
  float* ex_V = nullptr;    // [N][4]
  int ex_H = 0, ex_W = 0, ex_N = 0;
  bool ex_valid = false;
  // module-level WarpNet B-side cache
  bool warp_cache_valid = false;
  int warp_cache_sig[3] = {0, 0, 0};
  // correlation profiling
  bool prof_corr = false;
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> corr_events;
  // convolution profiling: per launch (start, stop, algorithmic FLOPs, kernel variant)
  bool prof_conv = false;
  struct ConvEv { cudaEvent_t e0, e1; double flops; int variant; };
  std::vector<ConvEv> conv_events;
};

static std::string g_create_err;

#define CUDA_TRY(ctx, expr)                                                                          \
  do {                                                                                                \
    cudaError_t e__ = (expr);                                                                         \
    if (e__ != cudaSuccess) {                                                                         \
      (ctx)->err = std::string(#expr) + ": " + cudaGetErrorString(e__);                              \
      return DVC_ERR_CUDA;                                                                            \
    }                                                                                                 \
  } while (0)

#define DVC_TRY(expr)          \
  do {                         \
    int r__ = (expr);          \
    if (r__ != DVC_OK) return r__; \
  } while (0)

static int fail(dvc_ctx* c, int code, const std::string& msg) {
  c->err = msg;
  return code;
}

// ------------------------------------------------------------------------------------------------
// buffers
// ------------------------------------------------------------------------------------------------
static int get_buf(dvc_ctx* c, const std::string& name, size_t bytes, void** out, const int sig[5], bool zero_on_change,
                   cudaStream_t s) {
  Buf& b = c->bufs[name];
  bool changed = false;
  if (b.bytes < bytes) {
    if (b.p) CUDA_TRY(c, cudaFree(b.p));
    b.p = nullptr;
    CUDA_TRY(c, cudaMalloc(&b.p, bytes));
    b.bytes = bytes;
    changed = true;
  }
  for (int i = 0; i < 5; ++i)
    if (b.sig[i] != sig[i]) changed = true, b.sig[i] = sig[i];
  if (changed && zero_on_change) CUDA_TRY(c, cudaMemsetAsync(b.p, 0, b.bytes, s));
  *out = b.p;
  return DVC_OK;
}

// padded NHWC activation; the zero border is established once per (name, shape) and never written by
// the convolution epilogues, the gather kernels rewrite their own borders every call.
// split: allocate tf32 hi/lo planes (input of a tensor-core convolution)
// mode 0: one fp32 plane; 1: tf32 hi/lo planes (fp32 words); 2: fp16 hi/lo planes of value * 2^e16 only;
// 3: an fp32 plane AND fp16 hi/lo planes (tensors that also feed a non-convolution consumer)
static int get_act(dvc_ctx* c, const std::string& name, int B, int H, int W, int C, int P, Act* a, cudaStream_t s,
                   int mode = 0) {
  *a = Act();
  a->B = B, a->H = H, a->W = W, a->C = C, a->P = P;
  const int sig[5] = {B, H, W, C, mode == 1 ? -1 - P : P + 1000 * mode};
  const size_t n = a->elems();
  const size_t bytes = mode == 0 ? n * 4 : (mode == 1 ? n * 8 : (mode == 2 ? n * 4 : n * 8));
  void* p = nullptr;
  DVC_TRY(get_buf(c, name, bytes, &p, sig, true, s));
  if (mode == 0 || mode == 1 || mode == 3) a->d = (float*)p;
  if (mode == 1) a->lo = a->d + n;
  if (mode == 2) a->h16 = p, a->l16 = (char*)p + n * 2;
  if (mode == 3) a->h16 = (char*)p + n * 4, a->l16 = (char*)p + n * 6;
  return DVC_OK;
}
static bool tc_mode(const dvc_ctx* c) { return c->conv_math == DVC_MATH_TF32X3; }

static int get_raw(dvc_ctx* c, const std::string& name, size_t bytes, void** out, cudaStream_t s) {
  const int sig[5] = {(int)(bytes & 0x7fffffff), 0, 0, 0, 0};
  return get_buf(c, name, bytes, out, sig, false, s);
}

// Two halves: [0] the frame-independent phase (VGG / WarpNet / correlation), [1] ColorVidNet -- the clip driver
// runs them concurrently on two streams, so they must not share statistics slots.
static int stats_begin(dvc_ctx* c, cudaStream_t s, int arena = 0) {
  const size_t need = 1 << 21;  // doubles (16 MB): far above the ~60 K used per forward at B <= 8
  if (c->stats_cap < need) {
    if (c->stats) CUDA_TRY(c, cudaFree(c->stats));
    CUDA_TRY(c, cudaMalloc((void**)&c->stats, need * sizeof(double)));
    c->stats_cap = need;
  }
  c->cur_arena = arena < 0 ? 0 : (arena > 2 ? 2 : arena);  // 0: phase A, 1: ColorVidNet, 2: phase A on the second stream
  c->stats_lo = (size_t)c->cur_arena * (need / 4);
  c->stats_hi = c->stats_lo + need / 4;
  c->stats_used = c->stats_lo;
  c->cell_left = 0;
  return DVC_OK;
}
static int stats_alloc(dvc_ctx* c, int B, int C, double** out, cudaStream_t s) {
  const size_t n = (size_t)B * C * 2;
  if (c->stats_used + n > c->stats_hi) return fail(c, DVC_ERR_STATE, "statistics arena exhausted (batch too large)");
  *out = c->stats + c->stats_used;
  c->stats_used += n;
  CUDA_TRY(c, cudaMemsetAsync(*out, 0, n * sizeof(double), s));
  return DVC_OK;
}

// device scale cells (dvc_internal.cuh: ScaleCell) come out of the statistics arena in chunks of 128, one memset each
static int cell_alloc(dvc_ctx* c, ScaleCell** out, cudaStream_t s) {
  if (c->cell_left == 0) {
    double* blk;
    DVC_TRY(stats_alloc(c, 1, 64, &blk, s));  // 128 doubles = 128 cells of 8 bytes
    c->cell_next = (ScaleCell*)blk, c->cell_left = 128;
  }
  *out = c->cell_next++;
  c->cell_left--;
  return DVC_OK;
}

static int check_launch(dvc_ctx* c, const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(c, DVC_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
  return DVC_OK;
}

// ------------------------------------------------------------------------------------------------
// weights
// ------------------------------------------------------------------------------------------------
static bool ends_with(const std::string& s, const char* suf) {
  const size_t n = strlen(suf);
  return s.size() >= n && s.compare(s.size() - n, n, suf) == 0;
}

// fp16 hi/lo planes of a packed [tap][cout][cin] weight block, scaled by the largest exact power of two that fits
static int upload_w16(dvc_ctx* c, const std::vector<float>& full, ConvW& w) {
  float amax = 0.f;
  for (float v : full) amax = fmaxf(amax, fabsf(v));
  w.e_w = e16_for(amax);
  {  // rows of `full` are [tap][cout][cin]: L1 norm per output channel
    const size_t cin = (size_t)w.cin_pad, cpt = (size_t)w.cout_pad_tc, taps = full.size() / (cin * cpt);
    std::vector<double> l1(cpt, 0.0);
    for (size_t t = 0; t < taps; ++t)
      for (size_t o = 0; o < cpt; ++o) {
        const float* r = &full[(t * cpt + o) * cin];
        double sacc = 0;
        for (size_t i = 0; i < cin; ++i) sacc += fabs((double)r[i]);
        l1[o] += sacc;
      }
    double m = 0;
    for (double v : l1) m = fmax(m, v);
    w.l1max = (float)(m * (1.0 + 1e-6));
  }
  std::vector<unsigned short> hi, lo;
  host_split16(full, w.e_w, hi, lo);
  if (w.w16_hi) cudaFree(w.w16_hi);
  if (w.w16_lo) cudaFree(w.w16_lo);
  w.w16_hi = w.w16_lo = nullptr;
  CUDA_TRY(c, cudaMalloc(&w.w16_hi, hi.size() * 2));
  CUDA_TRY(c, cudaMalloc(&w.w16_lo, lo.size() * 2));
  CUDA_TRY(c, cudaMemcpy(w.w16_hi, hi.data(), hi.size() * 2, cudaMemcpyHostToDevice));
  CUDA_TRY(c, cudaMemcpy(w.w16_lo, lo.data(), lo.size() * 2, cudaMemcpyHostToDevice));
  return DVC_OK;
}

extern "C" int dvc_set_weight(dvc_ctx* c, int net, const char* key_c, const float* data, const int64_t* shape,
                              int ndim) {
  if (!c || !key_c || !data || !shape || net < 0 || net > 2 || ndim < 1 || ndim > 4)
    return c ? fail(c, DVC_ERR_ARG, "dvc_set_weight: bad argument") : DVC_ERR_ARG;
  CUDA_TRY(c, cudaSetDevice(c->device));
  const std::string key(key_c);
  size_t n = 1;
  for (int i = 0; i < ndim; ++i) n *= (size_t)shape[i];
  std::vector<float> h(n);
  CUDA_TRY(c, cudaMemcpy(h.data(), data, n * sizeof(float), cudaMemcpyDefault));
  c->warp_cache_valid = false;
  c->ex_valid = c->ex_valid && net == DVC_NET_COLOR;  // exemplar operands depend on VGG/WarpNet weights

  if (ndim == 4 && ends_with(key, ".weight")) {
    const std::string base = key.substr(0, key.size() - 7);
    const int co = (int)shape[0], ci = (int)shape[1], kh = (int)shape[2], kw = (int)shape[3];
    if (ci == 1 && kh == 1 && kw == 1) {  // depthwise *_ss scale (ColorVidNet.py:12,16,21)
      float*& d = c->vec[net][base];
      if (d) cudaFree(d);
      CUDA_TRY(c, cudaMalloc((void**)&d, n * sizeof(float)));
      CUDA_TRY(c, cudaMemcpy(d, h.data(), n * sizeof(float), cudaMemcpyHostToDevice));
      float amax = 0.f;
      for (float v : h) amax = fmaxf(amax, fabsf(v));
      c->vec_absmax[net][base] = amax;
      return DVC_OK;
    }
    if (!((kh == 3 && kw == 3) || (kh == 1 && kw == 1))) return fail(c, DVC_ERR_SHAPE, "unsupported kernel size: " + key);
    if (co == 2 && kh == 1) {  // conv10_ab: consumed as [2][C] by the fused 1x1 + tanh kernel
      float*& d = c->vec[net][base];
      if (d) cudaFree(d);
      CUDA_TRY(c, cudaMalloc((void**)&d, n * sizeof(float)));
      CUDA_TRY(c, cudaMemcpy(d, h.data(), n * sizeof(float), cudaMemcpyHostToDevice));
    }
    ConvW& cw = c->conv[net][base];
    const int taps = kh * kw;
    const int cin_pad = (ci + 7) / 8 * 8;
    const int cout_pad = (co + 63) / 64 * 64;
    std::vector<float> packed((size_t)taps * cin_pad * cout_pad, 0.f);
    for (int o = 0; o < co; ++o)
      for (int i = 0; i < ci; ++i)
        for (int t = 0; t < taps; ++t)
          packed[((size_t)t * cin_pad + i) * cout_pad + o] = h[((size_t)o * ci + i) * taps + t];
    if (cw.w) cudaFree(cw.w);
    CUDA_TRY(c, cudaMalloc((void**)&cw.w, packed.size() * sizeof(float)));
    CUDA_TRY(c, cudaMemcpy(cw.w, packed.data(), packed.size() * sizeof(float), cudaMemcpyHostToDevice));
    if (!cw.b || cw.cout_pad != cout_pad) {
      if (cw.b) cudaFree(cw.b);
      CUDA_TRY(c, cudaMalloc((void**)&cw.b, cout_pad * sizeof(float)));
      CUDA_TRY(c, cudaMemset(cw.b, 0, cout_pad * sizeof(float)));
    }
    cw.cin = ci, cw.cin_pad = cin_pad, cw.cout = co, cw.cout_pad = cout_pad, cw.k = kh;
    {
      double m = 0;
      for (int o = 0; o < co; ++o) {
        double sacc = 0;
        for (size_t i = 0; i < (size_t)ci * taps; ++i) sacc += fabs((double)h[(size_t)o * ci * taps + i]);
        m = fmax(m, sacc);
      }
      cw.l1max = (float)(m * (1.0 + 1e-6));
    }
    if (cw.wt_hi) cudaFree(cw.wt_hi);
    if (cw.wt_lo) cudaFree(cw.wt_lo);
    cw.wt_hi = cw.wt_lo = nullptr;
    if (cin_pad % 32 == 0 && co >= 32) {  // tensor-core operand: [tap][cout_pad_tc][cin] hi / lo planes
      const int bn = conv_tc_pick_bn(co);
      const int cpt = (co + bn - 1) / bn * bn;
      std::vector<float> hi((size_t)taps * cpt * cin_pad, 0.f), lo(hi.size(), 0.f), full(hi.size(), 0.f);
      for (int o = 0; o < co; ++o)
        for (int i = 0; i < ci; ++i)
          for (int t = 0; t < taps; ++t) {
            const float v = h[((size_t)o * ci + i) * taps + t];
            const float vh = host_tf32_rna(v);
            full[((size_t)t * cpt + o) * cin_pad + i] = v;
            hi[((size_t)t * cpt + o) * cin_pad + i] = vh;
            lo[((size_t)t * cpt + o) * cin_pad + i] = host_tf32_rna(v - vh);
          }
      CUDA_TRY(c, cudaMalloc((void**)&cw.wt_hi, hi.size() * sizeof(float)));
      CUDA_TRY(c, cudaMalloc((void**)&cw.wt_lo, lo.size() * sizeof(float)));
      CUDA_TRY(c, cudaMemcpy(cw.wt_hi, hi.data(), hi.size() * sizeof(float), cudaMemcpyHostToDevice));
      CUDA_TRY(c, cudaMemcpy(cw.wt_lo, lo.data(), lo.size() * sizeof(float), cudaMemcpyHostToDevice));
      cw.cout_pad_tc = cpt;
      DVC_TRY(upload_w16(c, full, cw));
      if (net == DVC_NET_COLOR && taps == 9 && (base == "conv8_1.1" || base == "conv9_1.1" || base == "conv10_1.1")) {
        // ColorVidNet.py:81-83: Upsample(2, nearest) + Conv2d(3x3, pad 1).  Phase (a, b) of the output sees a 2x2
        // low-resolution neighbourhood whose weights are sums of the 3x3 taps that land on the same source pixel.
        for (int ph = 0; ph < 4; ++ph) {
          const int a = ph >> 1, b2 = ph & 1;
          ConvW& pw = c->conv[net][base + "#p" + std::to_string(ph)];
          std::vector<float> phi_((size_t)4 * cpt * cin_pad, 0.f), plo(phi_.size(), 0.f), pfull(phi_.size(), 0.f);
          for (int o = 0; o < co; ++o)
            for (int i = 0; i < ci; ++i)
              for (int r = 0; r < 2; ++r)
                for (int cc = 0; cc < 2; ++cc) {
                  float v = 0.f;
                  for (int ky = 0; ky < 3; ++ky) {
                    const bool rin = a ? (r == 0 ? ky <= 1 : ky == 2) : (r == 0 ? ky == 0 : ky >= 1);
                    if (!rin) continue;
                    for (int kx = 0; kx < 3; ++kx) {
                      const bool cin_ = b2 ? (cc == 0 ? kx <= 1 : kx == 2) : (cc == 0 ? kx == 0 : kx >= 1);
                      if (cin_) v += h[((size_t)o * ci + i) * 9 + ky * 3 + kx];
                    }
                  }
                  const float vh = host_tf32_rna(v);
                  pfull[((size_t)(r * 2 + cc) * cpt + o) * cin_pad + i] = v;
                  phi_[((size_t)(r * 2 + cc) * cpt + o) * cin_pad + i] = vh;
                  plo[((size_t)(r * 2 + cc) * cpt + o) * cin_pad + i] = host_tf32_rna(v - vh);
                }
          if (pw.wt_hi) cudaFree(pw.wt_hi);
          if (pw.wt_lo) cudaFree(pw.wt_lo);
          CUDA_TRY(c, cudaMalloc((void**)&pw.wt_hi, phi_.size() * sizeof(float)));
          CUDA_TRY(c, cudaMalloc((void**)&pw.wt_lo, plo.size() * sizeof(float)));
          CUDA_TRY(c, cudaMemcpy(pw.wt_hi, phi_.data(), phi_.size() * sizeof(float), cudaMemcpyHostToDevice));
          CUDA_TRY(c, cudaMemcpy(pw.wt_lo, plo.data(), plo.size() * sizeof(float), cudaMemcpyHostToDevice));
          pw.cin = ci, pw.cin_pad = cin_pad, pw.cout = co, pw.cout_pad = cout_pad, pw.cout_pad_tc = cpt, pw.k = 2;
          pw.cin_pad = cin_pad, pw.cout_pad_tc = cpt;
          DVC_TRY(upload_w16(c, pfull, pw));
          pw.b = nullptr;  // shares the bias of the 3x3 convolution (resolved at launch)
          pw.w = nullptr;
        }
      }
    }
    auto hb = c->host_bias[net].find(base);
    cw.bmax = 0.f;
    if (hb != c->host_bias[net].end()) {
      CUDA_TRY(c, cudaMemcpy(cw.b, hb->second.data(), hb->second.size() * sizeof(float), cudaMemcpyHostToDevice));
      for (float v : hb->second) cw.bmax = fmaxf(cw.bmax, fabsf(v));
    }
    return DVC_OK;
  }
  if (ndim == 1 && ends_with(key, ".bias")) {
    const std::string base = key.substr(0, key.size() - 5);
    c->host_bias[net][base] = h;
    auto it = c->conv[net].find(base);
    if (it != c->conv[net].end() && it->second.b) {
      if ((int)n > it->second.cout_pad) return fail(c, DVC_ERR_SHAPE, "bias longer than its weight: " + key);
      CUDA_TRY(c, cudaMemcpy(it->second.b, h.data(), n * sizeof(float), cudaMemcpyHostToDevice));
      it->second.bmax = 0.f;
      for (float v : h) it->second.bmax = fmaxf(it->second.bmax, fabsf(v));
    }
    if (base == "conv10_ab") {
      float*& d = c->vec[net]["conv10_ab.bias"];
      if (d) cudaFree(d);
      CUDA_TRY(c, cudaMalloc((void**)&d, n * sizeof(float)));
      CUDA_TRY(c, cudaMemcpy(d, h.data(), n * sizeof(float), cudaMemcpyHostToDevice));
    }
    return DVC_OK;
  }
  if (ndim == 1 && n == 1 && ends_with(key, ".weight")) {  // PReLU slope
    c->slope[net][key.substr(0, key.size() - 7)] = h[0];
    return DVC_OK;
  }
  return fail(c, DVC_ERR_ARG, "dvc_set_weight: unrecognised tensor " + key);
}

static int need_conv(dvc_ctx* c, int net, const char* name, const ConvW** out) {
  auto it = c->conv[net].find(name);
  if (it == c->conv[net].end() || !it->second.w)
    return fail(c, DVC_ERR_STATE, std::string("weight not set: ") + name + ".weight");
  if (c->host_bias[net].find(name) == c->host_bias[net].end())
    return fail(c, DVC_ERR_STATE, std::string("weight not set: ") + name + ".bias");
  *out = &it->second;
  return DVC_OK;
}
static int need_slope(dvc_ctx* c, int net, const char* name, float* out) {
  auto it = c->slope[net].find(name);
  if (it == c->slope[net].end()) return fail(c, DVC_ERR_STATE, std::string("weight not set: ") + name + ".weight");
  *out = it->second;
  return DVC_OK;
}
static int need_vec(dvc_ctx* c, int net, const char* name, const float** out) {
  auto it = c->vec[net].find(name);
  if (it == c->vec[net].end()) return fail(c, DVC_ERR_STATE, std::string("weight not set: ") + name);
  *out = it->second;
  return DVC_OK;
}

// ------------------------------------------------------------------------------------------------
// layer primitives
// ------------------------------------------------------------------------------------------------
struct ConvOpt {
  int dil = 1, stride = 1, act = ACT_NONE;
  int phase = -1;  // >= 0: phase (a*2+b) of a nearest-x2 + 3x3 convolution evaluated on the low-resolution input
  float slope = 0.f;
  const Act* add = nullptr;
  double* stats = nullptr;
  int yCoff = 0;
  const float* fin_w = nullptr;  // fused conv10_ab + tanh tail (tensor-core engine only): weights [2][Cout], bias [2],
  const float* fin_b = nullptr;  // NCHW destination [B][2][H][W]; the activated outputs themselves are not stored
  float* fin_out = nullptr;
  float l1_override = 0.f;  // > 0: weight L1 bound shared by the four phase launches of one up-convolution
};

// scale bookkeeping of a convolution whose output records max |y| (y.cell) and possibly stores fp16 planes (y.h16)
static int fill_dyn(dvc_ctx* c, const ConvW* w, const Act& x, const Act& y, const ConvOpt& o, DynOut* d) {
  *d = DynOut();
  if (x.cell) d->cell_in = x.cell;
  if (!y.cell) return DVC_OK;
  d->cell_out = y.cell;
  if (!y.h16) return DVC_OK;
  if (y.d) return fail(c, DVC_ERR_STATE, "conv: device-scaled output with an fp32 plane");
  d->h16 = y.h16, d->l16 = y.l16;
  if (!x.cell) d->in_bound = x.h16 ? ldexpf(32768.0f, -x.e16) : 0.f;
  if (!x.cell && !x.h16) return fail(c, DVC_ERR_STATE, "conv: device-scaled output needs a bounded input");
  if (o.add) {
    if (!o.add->cell) return fail(c, DVC_ERR_STATE, "conv: device-scaled output needs the addend's max");
    d->cell_add = o.add->cell;
  }
  d->w_l1 = o.l1_override > 0.f ? o.l1_override : w->l1max;
  d->b_max = w->bmax;
  d->gain = o.act == ACT_LRELU ? fmaxf(1.f, fabsf(o.slope)) : 1.f;
  return DVC_OK;
}

static int run_conv(dvc_ctx* c, const ConvW* w, const Act& x, Act& y, const ConvOpt& o, cudaStream_t s) {
  if (x.C != w->cin_pad) return fail(c, DVC_ERR_SHAPE, "conv: input channel mismatch");
  const int taps = o.phase >= 0 ? 4 : w->k * w->k;
  const bool f16 = x.h16 != nullptr;
  if (o.phase >= 0 && !x.lo && !f16) return fail(c, DVC_ERR_STATE, "conv: phase convolution needs the tensor-core engine");
  if (taps == 9 && x.P < o.dil) return fail(c, DVC_ERR_STATE, "conv: input border narrower than the dilation");
  ConvParams p{};
  p.x = x.d, p.Hp = x.Hp(), p.Wp = x.Wp(), p.P = x.P, p.H = x.H, p.W = x.W, p.Cin = x.C;
  p.w = w->w, p.bias = w->b, p.taps = taps, p.dil = o.dil, p.Cout = w->cout, p.CoutPad = w->cout_pad;
  p.stride = o.stride;
  p.Ho = (x.H + o.stride - 1) / o.stride, p.Wo = (x.W + o.stride - 1) / o.stride;
  if (o.phase >= 0) p.Ho = 2 * x.H, p.Wo = 2 * x.W;
  if (y.H != p.Ho || y.W != p.Wo || y.B != x.B || o.yCoff + w->cout > y.C)
    return fail(c, DVC_ERR_SHAPE, "conv: output shape mismatch");
  p.y = y.d, p.yHp = y.Hp(), p.yWp = y.Wp(), p.yP = y.P, p.yC = y.C, p.yCoff = o.yCoff;
  if (o.add) {
    if (o.add->H != p.Ho || o.add->W != p.Wo || o.add->C < w->cout) return fail(c, DVC_ERR_SHAPE, "conv: addend mismatch");
    p.add = o.add->d, p.aHp = o.add->Hp(), p.aWp = o.add->Wp(), p.aP = o.add->P, p.aC = o.add->C;
  }
  p.nchw = nullptr;
  p.act = o.act, p.slope = o.slope, p.stats = o.stats;
  p.y_lo = y.lo;
  if (x.lo || f16) {  // hi/lo planes: tensor-core engine (TF32 words, or fp16 halves of value * 2^e16)
    if (!w->wt_hi || (f16 && !w->w16_hi)) return fail(c, DVC_ERR_STATE, "conv: split input but no tensor-core weights");
    ConvTcParams t{};
    t.f16 = f16 ? 1 : 0;
    t.out_scale = f16 ? ldexpf(1.0f, -((x.cell ? 0 : x.e16) + w->e_w)) : 1.0f;
    if ((y.h16 || y.cell) && !f16) return fail(c, DVC_ERR_STATE, "conv: device-scaled outputs need the fp16 engine");
    DVC_TRY(fill_dyn(c, w, x, y, o, &t.dyn));
    t.Hp = p.Hp, t.Wp = p.Wp, t.P = p.P, t.H = p.H, t.W = p.W, t.Cin = p.Cin, t.Mtot = x.B * p.Hp * p.Wp;
    t.taps = taps, t.stride = o.stride, t.Cout = w->cout, t.CoutPad = w->cout_pad_tc, t.bias = w->b;
    t.oscale = 1, t.oa = 0, t.ob = 0;
    t.fin_w = o.fin_w, t.fin_b = o.fin_b, t.fin_out = o.fin_out;
    if (o.phase >= 0) {
      // nearest-x2 then 3x3 (zero pad 1) == four 2x2 convolutions on the low-resolution map, one per output parity
      // (a, b): rows {-1, 0} for a = 0 and {0, +1} for a = 1, same for columns (weights pre-summed at load time)
      const int a = o.phase >> 1, b2 = o.phase & 1;
      const int r0 = a ? 0 : -1, c0 = b2 ? 0 : -1;
      for (int r = 0; r < 2; ++r)
        for (int cc = 0; cc < 2; ++cc) t.tap_off[r * 2 + cc] = (r0 + r) * p.Wp + (c0 + cc);
      t.taps = 4, t.oscale = 2, t.oa = a, t.ob = b2;
    } else if (taps == 9) {
      for (int k = 0; k < 9; ++k) t.tap_off[k] = ((k / 3 - 1) * p.Wp + (k % 3 - 1)) * o.dil;
    } else {
      t.tap_off[0] = 0;
    }
    t.y = y.d, t.y_lo = y.lo, t.yHp = p.yHp, t.yWp = p.yWp, t.yP = p.yP, t.yC = p.yC, t.yCoff = p.yCoff;
    t.add = p.add, t.add_lo = o.add ? o.add->lo : nullptr, t.aHp = p.aHp, t.aWp = p.aWp, t.aP = p.aP, t.aC = p.aC;
    t.act = o.act, t.slope = o.slope, t.stats = o.stats, t.kc = c->tc_kc, t.cluster = c->tc_cluster, t.kbytes = c->tc_kbytes;
    t.tail = c->tc_tail;
    t.rowshare = c->tc_rowshare;
    t.dbg = c->tc_dbg;
    t.force_bn = (c->tc_force_bn && !o.fin_w && w->cout_pad_tc % c->tc_force_bn == 0) ? c->tc_force_bn : 0;
    t.splits = c->tc_splits, t.ws = nullptr, t.flags = nullptr, t.epoch = 0;
    if (c->tc_splits != 1 && (c->tc_splits > 1 || t.Mtot <= 128 * 8 * c->num_sms)) {  // split-K hand-over workspace + flags of this phase's arena (L2-resident, reused by every layer)
      const size_t mt = ((size_t)t.Mtot + 127) / 128 + 1;
      void *wsb, *flb;
      const int sigw[5] = {0, 0, 0, 0, 0};
      DVC_TRY(get_buf(c, "tc.ws" + std::to_string(c->cur_arena), mt * 128 * (size_t)w->cout_pad_tc * sizeof(float), &wsb, sigw, false, s));
      DVC_TRY(get_buf(c, "tc.flags" + std::to_string(c->cur_arena), (size_t)1 << 20, &flb, sigw, true, s));
      if (mt * (size_t)(w->cout_pad_tc / 64) < ((size_t)1 << 18)) {
        t.ws = (float*)wsb, t.flags = (int*)flb, t.epoch = ++c->tc_epoch[c->cur_arena];
      }
    }
    std::string err;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    if (c->prof_conv) {
      CUDA_TRY(c, cudaEventCreate(&e0));
      CUDA_TRY(c, cudaEventCreate(&e1));
      CUDA_TRY(c, cudaEventRecord(e0, s));
    }
    int variant = 0;
    const int lrc = f16 ? launch_conv_tc(t, x.h16, x.l16, w->w16_hi, w->w16_lo, c->num_sms, s, &err, &variant)
                        : launch_conv_tc(t, x.d, x.lo, w->wt_hi, w->wt_lo, c->num_sms, s, &err, &variant);
    if (lrc != 0) return fail(c, DVC_ERR_CUDA, "conv_tc: " + err);
    if (c->prof_conv) {
      CUDA_TRY(c, cudaEventRecord(e1, s));
      // algorithmic FLOPs: 2 x output pixels x taps x Cin x Cout (padding channels and masked border pixels excluded)
      c->conv_events.push_back({e0, e1, 2.0 * x.B * (o.phase >= 0 ? x.H * x.W : p.Ho * p.Wo) * taps * (double)w->cin * w->cout, variant});
    }
    return check_launch(c, "conv_tc");
  }
  if (o.add && o.add->lo) return fail(c, DVC_ERR_STATE, "conv: CUDA-core kernel cannot read a split addend");
  // tensor-core mode: the two K = 27 / 63 first layers use the per-pixel kernel (the fp32 parity mode keeps the
  // two-level GEMM kernel for every layer)
  if (y.h16 || y.cell) {
    if (!x.cell) return fail(c, DVC_ERR_STATE, "conv: first layer needs the input's max");
    DVC_TRY(fill_dyn(c, w, x, y, o, &p.dyn));
    if (!launch_conv_first(p, x.B, w->cin, s)) return fail(c, DVC_ERR_STATE, "conv: device-scaled outputs need the first-layer kernel");
    return check_launch(c, "conv_first");
  }
  if (tc_mode(c) && launch_conv_first(p, x.B, w->cin, s)) return check_launch(c, "conv_first");
  launch_conv_simt(p, x.B, c->two_level, s);
  return check_launch(c, "conv");
}

struct XfOpt {
  int pad_mode = PAD_ZERO, up = 1, sub = 1, rowpad = 0;
  const double* stats = nullptr;
  double count = 1.0;
  const float* scale = nullptr;
  const Act* res = nullptr;
  int act = 0;
  float slope = 0.f;
  int dCoff = 0, C = 0;
};

static int run_xform(dvc_ctx* c, const Act& src, Act& dst, const XfOpt& o, cudaStream_t s) {
  const int C = o.C ? o.C : src.C;
  const int eh = ((src.H + o.sub - 1) / o.sub) * o.up + 2 * o.rowpad, ew = ((src.W + o.sub - 1) / o.sub) * o.up;
  if (dst.H != eh || dst.W != ew || dst.B != src.B || o.dCoff + C > dst.C || (C & 7) || (o.dCoff & 7) || (dst.C & 7) || (src.C & 7))
    return fail(c, DVC_ERR_SHAPE, "xform: shape mismatch");
  if (o.pad_mode == PAD_REFLECT && (dst.P >= dst.H || dst.P >= dst.W)) return fail(c, DVC_ERR_SHAPE, "xform: reflect pad too wide");
  XformParams p{};
  p.src = src.d, p.src_lo = src.lo, p.sH = src.H, p.sW = src.W, p.sP = src.P, p.sC = src.C, p.sCoff = 0;
  p.dst_lo = dst.lo;
  p.dst_h16 = dst.h16, p.dst_l16 = dst.l16, p.dscale16 = ldexpf(1.0f, dst.e16);
  p.dst = dst.d, p.dH = dst.H, p.dW = dst.W, p.dP = dst.P, p.dC = dst.C, p.dCoff = o.dCoff;
  p.C = C, p.pad_mode = o.pad_mode, p.up = o.up, p.sub = o.sub, p.rowpad = o.rowpad;
  p.stats = o.stats, p.count = o.count, p.eps = 1e-5f, p.scale = o.scale;
  if (o.res) {
    if (o.res->H != dst.H || o.res->W != dst.W || o.res->C < C) return fail(c, DVC_ERR_SHAPE, "xform: residual mismatch");
    p.res = o.res->d, p.res_lo = o.res->lo, p.rP = o.res->P, p.rC = o.res->C;
  }
  p.act = o.act, p.slope = o.slope;
  launch_xform(p, src.B, s);
  return check_launch(c, "xform");
}

static int run_pixnorm(dvc_ctx* c, const Act& src, float* dst, float* dst_lo, int dP, int pad_mode, const double* stats,
                       double count, cudaStream_t s, void* h16 = nullptr, void* l16 = nullptr, int e16 = 0) {
  if (src.C != 128 && src.C != 256 && src.C != 512) return fail(c, DVC_ERR_SHAPE, "pixnorm: channel count");
  PixNormParams p{};
  p.src = src.d, p.src_lo = src.lo, p.sH = src.H, p.sW = src.W, p.sP = src.P, p.sC = src.C;
  if (src.h16 && !src.d) {
    if (!src.cell) return fail(c, DVC_ERR_STATE, "pixnorm: fp16 source without a scale cell");
    p.src_h16 = src.h16, p.src_l16 = src.l16, p.src_cell = src.cell;
  }
  p.dst = dst, p.dst_lo = dst_lo, p.dP = dP, p.dC = src.C, p.C = src.C, p.pad_mode = pad_mode;
  p.dst_h16 = h16, p.dst_l16 = l16, p.dscale16 = ldexpf(1.0f, e16);
  p.stats = stats, p.count = count, p.eps = 2.220446049250313e-16f;  // sys.float_info.epsilon
  launch_pixnorm(p, src.B, s);
  return check_launch(c, "pixnorm");
}

// ------------------------------------------------------------------------------------------------
// VGG19 trunk (NonlocalNet.py:228-256)
// ------------------------------------------------------------------------------------------------
struct VggMaps {
  std::map<std::string, Act> m;  // "r11".."r54", "p1".."p5"
};

static const char* kVggSeq[] = {"conv1_1", "conv1_2", "P", "conv2_1", "conv2_2", "P", "conv3_1", "conv3_2", "conv3_3",
                                "conv3_4", "P", "conv4_1", "conv4_2", "conv4_3", "conv4_4", "P", "conv5_1", "conv5_2",
                                "conv5_3", "conv5_4", "P"};

// x0: padded NHWC, 8 channels (3 used), P=1.  Runs until `last_key` has been produced.
static int vgg_trunk(dvc_ctx* c, const std::string& tag, const Act& x0, const std::string& last_key, VggMaps* out,
                     cudaStream_t s) {
  Act cur = x0;
  // tensor-core mode: the whole conv -> ReLU -> conv trunk lives on fp16 hi/lo planes whose exact power-of-two scale
  // each layer derives on the device from the measured max |input| and its weights' L1 norm (DynOut)
  const bool dyn = tc_mode(c) && c->tc_f16;
  const int mode = dyn ? 2 : (tc_mode(c) ? 1 : 0);
  if (dyn) {
    DVC_TRY(cell_alloc(c, &cur.cell, s));
    launch_amax(cur.d, cur.elems(), cur.cell, s);
    DVC_TRY(check_launch(c, "amax"));
  }
  int block = 1, idx = 1;
  for (const char* name : kVggSeq) {
    std::string key;
    Act nxt;
    if (name[0] == 'P') {
      key = "p" + std::to_string(block);
      DVC_TRY(get_act(c, tag + "." + key, cur.B, cur.H / 2, cur.W / 2, cur.C, 1, &nxt, s, mode));
      if (dyn) {
        DVC_TRY(cell_alloc(c, &nxt.cell, s));
        launch_maxpool2_h16(cur.h16, cur.l16, cur.cell, cur.H, cur.W, cur.P, cur.C, nxt.h16, nxt.l16, nxt.cell, 1, cur.B, s);
      } else {
        launch_maxpool2(cur.d, cur.lo, cur.H, cur.W, cur.P, cur.C, nxt.d, nxt.lo, 1, cur.B, s);
      }
      DVC_TRY(check_launch(c, "maxpool"));
      block++, idx = 1;
    } else {
      key = "r" + std::to_string(block) + std::to_string(idx);
      const ConvW* w;
      DVC_TRY(need_conv(c, DVC_NET_VGG, name, &w));
      DVC_TRY(get_act(c, tag + "." + key, cur.B, cur.H, cur.W, w->cout, 1, &nxt, s, mode));
      if (dyn) DVC_TRY(cell_alloc(c, &nxt.cell, s));
      ConvOpt o;
      o.act = ACT_RELU;
      DVC_TRY(run_conv(c, w, cur, nxt, o, s));
      idx++;
    }
    out->m[key] = nxt;
    cur = nxt;
    if (key == last_key) break;
    if (cur.H < 2 || cur.W < 2) break;
  }
  return DVC_OK;
}

// ------------------------------------------------------------------------------------------------
// WarpNet feature side (NonlocalNet.py:451-476 for one of A / B)
// ------------------------------------------------------------------------------------------------
// n[4]: normalised r22,r32,r42,r52 maps, reflect-padded (P=1).  Writes rows [B][N][256] to `rows_out`.
static int warp_side(dvc_ctx* c, const std::string& tag, const Act n[4], const char* proj, float* rows_out, int h, int w,
                     cudaStream_t s) {
  const int net = DVC_NET_WARP;
  const int B = n[0].B;
  Act cat;
  // tensor-core mode: every tensor below is an InstanceNorm output (|z| <= sqrt(count)) through a PReLU, so its fp16
  // hi/lo planes get a static exact power-of-two scale; cat and the residual chain also keep an fp32 plane (mode 3)
  const bool h16 = tc_mode(c) && c->tc_f16;
  const int sp = h16 ? 2 : (tc_mode(c) ? 1 : 0), sp_res = h16 ? 3 : sp;
  DVC_TRY(get_act(c, tag + ".cat", B, h, w, 256, 1, &cat, s, sp_res));

  struct Head {
    const char* c1;
    const char* s1;
    const char* c2;
    const char* s2;
    int stride2, up_mid, up_end;
  };
  const Head heads[4] = {{"layer2_1.1", "layer2_1.3", "layer2_1.5", "layer2_1.7", 2, 1, 1},
                         {"layer3_1.1", "layer3_1.3", "layer3_1.5", "layer3_1.7", 1, 1, 1},
                         {"layer4_1.1", "layer4_1.3", "layer4_1.5", "layer4_1.7", 1, 1, 2},
                         {"layer5_1.1", "layer5_1.3", "layer5_1.6", "layer5_1.8", 1, 2, 2}};
  double cat_bound = 0;  // every head's last InstanceNorm runs over at most h*w positions
  for (int k = 0; k < 4; ++k) {
    float s2;
    DVC_TRY(need_slope(c, net, heads[k].s2, &s2));
    cat_bound = fmax(cat_bound, sqrt((double)h * w) * fmax(1.0, fabs(s2)));
  }
  cat.e16 = e16_for(cat_bound);
  for (int k = 0; k < 4; ++k) {
    const Head& hd = heads[k];
    const ConvW *w1, *w2;
    float s1, s2;
    DVC_TRY(need_conv(c, net, hd.c1, &w1));
    DVC_TRY(need_conv(c, net, hd.c2, &w2));
    DVC_TRY(need_slope(c, net, hd.s1, &s1));
    DVC_TRY(need_slope(c, net, hd.s2, &s2));
    const std::string t = tag + ".h" + std::to_string(k);
    const Act& x = n[k];
    Act raw1, mid, raw2;
    double *st1, *st2;
    DVC_TRY(get_act(c, t + ".raw1", B, x.H, x.W, w1->cout, 0, &raw1, s));
    DVC_TRY(stats_alloc(c, B, w1->cout, &st1, s));
    ConvOpt o1;
    o1.stats = st1;
    DVC_TRY(run_conv(c, w1, x, raw1, o1, s));
    DVC_TRY(get_act(c, t + ".mid", B, x.H * hd.up_mid, x.W * hd.up_mid, w1->cout, 1, &mid, s, sp));
    mid.e16 = e16_for(sqrt((double)x.H * x.W) * fmax(1.0, fabs(s1)));
    XfOpt x1;
    x1.pad_mode = PAD_REFLECT, x1.up = hd.up_mid, x1.stats = st1, x1.count = (double)x.H * x.W, x1.act = 2, x1.slope = s1;
    DVC_TRY(run_xform(c, raw1, mid, x1, s));
    const int h2 = (mid.H + hd.stride2 - 1) / hd.stride2, w2o = (mid.W + hd.stride2 - 1) / hd.stride2;

    DVC_TRY(get_act(c, t + ".raw2", B, h2, w2o, 64, 0, &raw2, s));
    DVC_TRY(stats_alloc(c, B, 64, &st2, s));
    ConvOpt o2;
    o2.stats = st2, o2.stride = hd.stride2;
    DVC_TRY(run_conv(c, w2, mid, raw2, o2, s));
    XfOpt x2;
    x2.pad_mode = PAD_REFLECT, x2.up = hd.up_end, x2.stats = st2, x2.count = (double)h2 * w2o, x2.act = 2, x2.slope = s2;
    x2.dCoff = 64 * k, x2.C = 64;
    const int fh = h2 * hd.up_end, fw = w2o * hd.up_end;
    if (fw != w) return fail(c, DVC_ERR_SHAPE, "WarpNet: feature widths disagree (W must be a multiple of 16)");
    if (fh != h) {
      // NonlocalNet.py:461-463 repairs only the r5 head, rows only, by exactly one row top and bottom
      if (k != 3 || fh + 2 != h) return fail(c, DVC_ERR_SHAPE, "WarpNet: feature heights disagree (H must be a multiple of 8)");
      x2.rowpad = 1;
    }
    DVC_TRY(run_xform(c, raw2, cat, x2, s));
  }

  // three residual blocks (NonlocalNet.py:341-352), ping-pong between two padded buffers
  Act xa = cat, xb, raw, mid;
  DVC_TRY(get_act(c, tag + ".res_b", B, h, w, 256, 1, &xb, s, sp_res));
  DVC_TRY(get_act(c, tag + ".res_raw", B, h, w, 256, 0, &raw, s));
  DVC_TRY(get_act(c, tag + ".res_mid", B, h, w, 256, 1, &mid, s, sp));
  double chain_bound = cat_bound;
  for (int i = 0; i < 3; ++i) {
    const std::string base = "layer." + std::to_string(i);
    const ConvW *w1, *w2;
    float sl;
    DVC_TRY(need_conv(c, net, (base + ".conv1").c_str(), &w1));
    DVC_TRY(need_conv(c, net, (base + ".conv2").c_str(), &w2));
    DVC_TRY(need_slope(c, net, (base + ".prelu").c_str(), &sl));
    double *st1, *st2;
    DVC_TRY(stats_alloc(c, B, 256, &st1, s));
    DVC_TRY(stats_alloc(c, B, 256, &st2, s));
    ConvOpt o1;
    o1.stats = st1;
    DVC_TRY(run_conv(c, w1, xa, raw, o1, s));
    XfOpt x1;
    x1.pad_mode = PAD_REFLECT, x1.stats = st1, x1.count = (double)h * w, x1.act = 2, x1.slope = sl;
    const double in_bound = sqrt((double)h * w) * fmax(1.0, fabs(sl));
    mid.e16 = e16_for(in_bound);
    DVC_TRY(run_xform(c, raw, mid, x1, s));
    ConvOpt o2;
    o2.stats = st2;
    DVC_TRY(run_conv(c, w2, mid, raw, o2, s));
    XfOpt x2;
    x2.pad_mode = PAD_REFLECT, x2.stats = st2, x2.count = (double)h * w, x2.act = 2, x2.slope = sl, x2.res = &xa;
    // out = PReLU(IN(conv2(..)) + x) (NonlocalNet.py:341-352): |out| <= (sqrt(hw) + |x|max) * max(1, |slope|)
    chain_bound = (chain_bound + sqrt((double)h * w)) * fmax(1.0, fabs(sl));
    xb.e16 = e16_for(chain_bound);
    DVC_TRY(run_xform(c, raw, xb, x2, s));
    std::swap(xa, xb);
  }

  // theta / phi: 1x1 conv, centre over positions, unit L2 norm over channels (NonlocalNet.py:468-476)
  const ConvW* wp;
  DVC_TRY(need_conv(c, net, proj, &wp));
  double* stp;
  DVC_TRY(stats_alloc(c, B, 256, &stp, s));
  ConvOpt op;
  op.stats = stp;
  DVC_TRY(run_conv(c, wp, xa, raw, op, s));
  DVC_TRY(run_pixnorm(c, raw, rows_out, nullptr, 0, PAD_ZERO, stp, (double)h * w, s));
  return DVC_OK;
}

// ------------------------------------------------------------------------------------------------
// correlation dispatch
// ------------------------------------------------------------------------------------------------
static int run_corr(dvc_ctx* c, const CorrParams& p, cudaStream_t s, long long phi_version = -1, CorrWorkspace* ws = nullptr) {
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  if (c->prof_corr) {
    CUDA_TRY(c, cudaEventCreate(&e0));
    CUDA_TRY(c, cudaEventCreate(&e1));
    CUDA_TRY(c, cudaEventRecord(e0, s));
  }
  if (c->corr_math == DVC_MATH_FP32) {
    launch_corr_simt(p, s);
  } else {
    std::string err;
    if (launch_corr_tc(p, c->corr_math, c->corr_cluster, c->corr_screen, ws ? ws : &c->corr_ws, phi_version, s, &err) != 0)
      return fail(c, DVC_ERR_CUDA, "corr_tc: " + err);
  }
  DVC_TRY(check_launch(c, "corr"));
  if (c->prof_corr) {
    CUDA_TRY(c, cudaEventRecord(e1, s));
    c->corr_events.emplace_back(e0, e1);
  }
  return DVC_OK;
}

// ------------------------------------------------------------------------------------------------
// ColorVidNet (ColorVidNet.py:96-144).  in0: padded NHWC, 8 channels (7 used), P=1, zero border.
// ------------------------------------------------------------------------------------------------
static int colorvid(dvc_ctx* c, const std::string& tag, const Act& in0, float* out_nchw, cudaStream_t s) {
  const int net = DVC_NET_COLOR;
  const int B = in0.B, H = in0.H, W = in0.W;
  int uid = 0;
  const bool dyn = tc_mode(c) && c->tc_f16;
  auto conv = [&](const char* name, const Act& x, Act* y, int outP, int act, int dil, const Act* add, double** st,
                  float slope) -> int {
    const ConvW* w;
    DVC_TRY(need_conv(c, net, name, &w));
    // outputs with a border (outP > 0) feed another convolution: hi/lo planes in tensor-core mode
    // ... fp16 planes with a device-derived scale when the fp16 engine is on (conv -> ReLU -> conv chains)
    const bool tcx = x.lo || x.h16;  // this launch runs on the tensor-core engine
    DVC_TRY(get_act(c, tag + "." + name + "#" + std::to_string(uid++), x.B, x.H, x.W, w->cout, outP, y, s,
                    (tc_mode(c) && outP > 0) ? (dyn ? 2 : 1) : 0));
    if (dyn && (tcx || outP > 0)) DVC_TRY(cell_alloc(c, &y->cell, s));
    ConvOpt o;
    o.act = act, o.dil = dil, o.add = add, o.slope = slope;
    if (st) {
      DVC_TRY(stats_alloc(c, B, w->cout, st, s));
      o.stats = *st;
    }
    return run_conv(c, w, x, *y, o, s);
  };
  // InstanceNorm outputs are bounded by sqrt(count) (x |scale|): fp16 hi/lo planes with a static power-of-two scale
  auto norm = [&](const char* name, const Act& raw, const double* st, Act* y, int outP, int up, int sub,
                  const float* scale, float scale_abs = 1.f) -> int {
    DVC_TRY(get_act(c, tag + "." + name + "#" + std::to_string(uid++), B, ((raw.H + sub - 1) / sub) * up,
                    ((raw.W + sub - 1) / sub) * up, raw.C, outP, y, s, tc_mode(c) ? (c->tc_f16 ? 2 : 1) : 0));
    y->e16 = e16_for(sqrt((double)raw.H * raw.W) * fmax(1e-3, (double)scale_abs));
    XfOpt o;
    o.pad_mode = PAD_ZERO, o.up = up, o.sub = sub, o.stats = st, o.count = (double)raw.H * raw.W, o.scale = scale;
    return run_xform(c, raw, *y, o, s);
  };
  // decoder "deconv" = nearest x2 + 3x3 conv (ColorVidNet.py:81-83) + skip add + ReLU.  Tensor-core mode evaluates
  // it as four 2x2 phase convolutions on the low-resolution map (2.25x fewer MACs, no up-sampled activation in HBM);
  // the CUDA-core mode keeps the literal formulation.
  auto upconv = [&](const char* name, const Act& raw, const double* st, const Act* add, Act* y) -> int {
    const ConvW* w;
    DVC_TRY(need_conv(c, net, name, &w));
    DVC_TRY(get_act(c, tag + "." + name + "#" + std::to_string(uid++), B, raw.H * 2, raw.W * 2, w->cout, 1, y, s,
                    tc_mode(c) ? (dyn ? 2 : 1) : 0));
    if (tc_mode(c)) {
      Act nl;
      DVC_TRY(norm((std::string(name) + ".in").c_str(), raw, st, &nl, 1, 1, 1, nullptr));
      float l1 = 0.f;  // one exponent for the four phases that fill the same tensor
      if (dyn) {
        DVC_TRY(cell_alloc(c, &y->cell, s));
        for (int ph = 0; ph < 4; ++ph) {
          auto it = c->conv[net].find(std::string(name) + "#p" + std::to_string(ph));
          if (it != c->conv[net].end()) l1 = fmaxf(l1, it->second.l1max);
        }
      }
      for (int ph = 0; ph < 4; ++ph) {
        auto it = c->conv[net].find(std::string(name) + "#p" + std::to_string(ph));
        if (it == c->conv[net].end() || !it->second.wt_hi || !it->second.w16_hi) return fail(c, DVC_ERR_STATE, std::string("phase weights missing: ") + name);
        ConvW pw = it->second;
        pw.b = w->b, pw.bmax = w->bmax;
        ConvOpt o;
        o.act = ACT_RELU, o.add = add, o.phase = ph, o.l1_override = l1;
        DVC_TRY(run_conv(c, &pw, nl, *y, o, s));
      }
      return DVC_OK;
    }
    Act nu;
    DVC_TRY(norm((std::string(name) + ".in").c_str(), raw, st, &nu, 1, 2, 1, nullptr));
    ConvOpt o;
    o.act = ACT_RELU, o.add = add;
    return run_conv(c, w, nu, *y, o, s);
  };
  const float *ss1, *ss2, *ss3, *wab, *bab;
  DVC_TRY(need_vec(c, net, "conv1_2norm_ss", &ss1));
  DVC_TRY(need_vec(c, net, "conv2_2norm_ss", &ss2));
  DVC_TRY(need_vec(c, net, "conv3_3norm_ss", &ss3));
  DVC_TRY(need_vec(c, net, "conv10_ab", &wab));
  DVC_TRY(need_vec(c, net, "conv10_ab.bias", &bab));

  Act a, b, raw1, n1, d1, raw2, n2, d2, raw3, n3, d3, raw4, n4, raw5, n5, raw6, n6, raw7, t, u;
  double *st1, *st2, *st3, *st4, *st5, *st6, *st7, *st8, *st9;
  Act xin = in0;
  if (dyn) {
    DVC_TRY(cell_alloc(c, &xin.cell, s));
    launch_amax(xin.d, xin.elems(), xin.cell, s);
    DVC_TRY(check_launch(c, "amax"));
  }
  DVC_TRY(conv("conv1_1.0", xin, &a, 1, ACT_RELU, 1, nullptr, nullptr, 0));
  DVC_TRY(conv("conv1_1.2", a, &b, 1, ACT_RELU, 1, nullptr, nullptr, 0));
  DVC_TRY(conv("conv1_2", b, &raw1, 0, ACT_RELU, 1, nullptr, &st1, 0));
  DVC_TRY(norm("n1", raw1, st1, &n1, 1, 1, 1, nullptr));
  DVC_TRY(norm("d1", raw1, st1, &d1, 1, 1, 2, ss1, c->vec_absmax[net]["conv1_2norm_ss"]));
  DVC_TRY(conv("conv2_1", d1, &a, 1, ACT_RELU, 1, nullptr, nullptr, 0));
  DVC_TRY(conv("conv2_2", a, &raw2, 0, ACT_RELU, 1, nullptr, &st2, 0));
  DVC_TRY(norm("n2", raw2, st2, &n2, 1, 1, 1, nullptr));
  DVC_TRY(norm("d2", raw2, st2, &d2, 1, 1, 2, ss2, c->vec_absmax[net]["conv2_2norm_ss"]));
  DVC_TRY(conv("conv3_1", d2, &a, 1, ACT_RELU, 1, nullptr, nullptr, 0));
  DVC_TRY(conv("conv3_2", a, &b, 1, ACT_RELU, 1, nullptr, nullptr, 0));
  DVC_TRY(conv("conv3_3", b, &raw3, 0, ACT_RELU, 1, nullptr, &st3, 0));
  DVC_TRY(norm("n3", raw3, st3, &n3, 1, 1, 1, nullptr));
  DVC_TRY(norm("d3", raw3, st3, &d3, 1, 1, 2, ss3, c->vec_absmax[net]["conv3_3norm_ss"]));
  DVC_TRY(conv("conv4_1", d3, &a, 1, ACT_RELU, 1, nullptr, nullptr, 0));
  DVC_TRY(conv("conv4_2", a, &b, 1, ACT_RELU, 1, nullptr, nullptr, 0));
  DVC_TRY(conv("conv4_3", b, &raw4, 0, ACT_RELU, 1, nullptr, &st4, 0));
  DVC_TRY(norm("n4", raw4, st4, &n4, 2, 1, 1, nullptr));
  DVC_TRY(conv("conv5_1", n4, &a, 2, ACT_RELU, 2, nullptr, nullptr, 0));
  DVC_TRY(conv("conv5_2", a, &b, 2, ACT_RELU, 2, nullptr, nullptr, 0));
  DVC_TRY(conv("conv5_3", b, &raw5, 0, ACT_RELU, 2, nullptr, &st5, 0));
  DVC_TRY(norm("n5", raw5, st5, &n5, 2, 1, 1, nullptr));
  DVC_TRY(conv("conv6_1", n5, &a, 2, ACT_RELU, 2, nullptr, nullptr, 0));
  DVC_TRY(conv("conv6_2", a, &b, 2, ACT_RELU, 2, nullptr, nullptr, 0));
  DVC_TRY(conv("conv6_3", b, &raw6, 0, ACT_RELU, 2, nullptr, &st6, 0));
  DVC_TRY(norm("n6", raw6, st6, &n6, 1, 1, 1, nullptr));
  DVC_TRY(conv("conv7_1", n6, &a, 1, ACT_RELU, 1, nullptr, nullptr, 0));
  DVC_TRY(conv("conv7_2", a, &b, 1, ACT_RELU, 1, nullptr, nullptr, 0));
  DVC_TRY(conv("conv7_3", b, &raw7, 0, ACT_RELU, 1, nullptr, &st7, 0));
  // decoder stage 8: relu(conv8_1(up(n7)) + conv3_3_short(n3))
  DVC_TRY(conv("conv3_3_short", n3, &t, 0, ACT_NONE, 1, nullptr, nullptr, 0));
  DVC_TRY(upconv("conv8_1.1", raw7, st7, &t, &u));
  DVC_TRY(conv("conv8_2", u, &a, 1, ACT_RELU, 1, nullptr, nullptr, 0));
  DVC_TRY(conv("conv8_3", a, &raw1, 0, ACT_RELU, 1, nullptr, &st8, 0));
  DVC_TRY(conv("conv2_2_short", n2, &t, 0, ACT_NONE, 1, nullptr, nullptr, 0));
  DVC_TRY(upconv("conv9_1.1", raw1, st8, &t, &u));
  DVC_TRY(conv("conv9_2", u, &raw2, 0, ACT_RELU, 1, nullptr, &st9, 0));
  DVC_TRY(conv("conv1_2_short", n1, &t, 0, ACT_NONE, 1, nullptr, nullptr, 0));
  DVC_TRY(upconv("conv10_1.1", raw2, st9, &t, &u));
  if (u.H != H || u.W != W) return fail(c, DVC_ERR_SHAPE, "ColorVidNet: decoder shape mismatch");
  if (tc_mode(c) && (u.lo || u.h16)) {
    // conv10_2 + LeakyReLU(0.2) + conv10_ab (1x1, 128 -> 2) + tanh * 128 in one launch: the 128-channel full-resolution
    // activation (213 MB at 480p) is consumed in the epilogue instead of being written and re-read
    const ConvW* w;
    DVC_TRY(need_conv(c, net, "conv10_2", &w));
    if (w->cout != 128) return fail(c, DVC_ERR_SHAPE, "ColorVidNet: conv10_2 must have 128 output channels");
    Act none;
    none.B = B, none.H = H, none.W = W, none.C = w->cout, none.P = 0;
    ConvOpt o;
    o.act = ACT_LRELU, o.slope = 0.2f, o.fin_w = wab, o.fin_b = bab, o.fin_out = out_nchw;
    return run_conv(c, w, u, none, o, s);
  }
  DVC_TRY(conv("conv10_2", u, &a, 0, ACT_LRELU, 1, nullptr, nullptr, 0.2f));
  if (a.H != H || a.W != W || a.C != 128) return fail(c, DVC_ERR_SHAPE, "ColorVidNet: decoder shape mismatch");
  launch_final_ab(a.d, H, W, a.P, a.C, wab, bab, out_nchw, B, s);
  return check_launch(c, "final_ab");
}

// ------------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------------
static bool legal_shape(int H, int W) { return H >= 16 && W >= 16 && H % 8 == 0 && W % 16 == 0; }

extern "C" const char* dvc_version(void) { return "libdvc 0.1 (sm_100a)"; }

extern "C" int dvc_create(dvc_ctx** out, int device) {
  if (!out) return DVC_ERR_ARG;
  *out = nullptr;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0) {
    g_create_err = std::string("no CUDA device: ") + cudaGetErrorString(e) + " (libdvc has no CPU fallback)";
    return DVC_ERR_CUDA;
  }
  if (device < 0 || device >= n) {
    g_create_err = "device index out of range";
    return DVC_ERR_ARG;
  }
  e = cudaSetDevice(device);
  if (e != cudaSuccess) {
    g_create_err = cudaGetErrorString(e);
    return DVC_ERR_CUDA;
  }
  cudaDeviceProp prop;
  cudaGetDeviceProperties(&prop, device);
  if (prop.major != 10) {
    g_create_err = "libdvc is built for sm_100a only; device is sm_" + std::to_string(prop.major * 10 + prop.minor);
    return DVC_ERR_CUDA;
  }
  dvc_ctx* c = new dvc_ctx();
  c->device = device;
  c->num_sms = prop.multiProcessorCount;
  *out = c;
  return DVC_OK;
}

extern "C" int dvc_destroy(dvc_ctx* c) {
  if (!c) return DVC_ERR_ARG;
  cudaSetDevice(c->device);
  cudaDeviceSynchronize();
  for (auto& kv : c->bufs)
    if (kv.second.p) cudaFree(kv.second.p);
  for (int n = 0; n < 3; ++n) {
    for (auto& kv : c->conv[n]) {
      if (kv.second.w) cudaFree(kv.second.w);
      if (kv.second.b) cudaFree(kv.second.b);
      if (kv.second.wt_hi) cudaFree(kv.second.wt_hi);
      if (kv.second.w16_hi) cudaFree(kv.second.w16_hi);
      if (kv.second.w16_lo) cudaFree(kv.second.w16_lo);
      if (kv.second.wt_lo) cudaFree(kv.second.wt_lo);
    }
    for (auto& kv : c->vec[n])
      if (kv.second) cudaFree(kv.second);
  }
  if (c->stats) cudaFree(c->stats);
  if (c->sA) cudaStreamDestroy(c->sA);
  if (c->sA2) cudaStreamDestroy(c->sA2);
  if (c->evJoinA2) cudaEventDestroy(c->evJoinA2);
  corr_ws_free(&c->corr_ws2);
  if (c->sC) cudaStreamDestroy(c->sC);
  for (int i = 0; i < 4; ++i) {
    if (c->evA[i]) cudaEventDestroy(c->evA[i]);
    if (c->evU[i]) cudaEventDestroy(c->evU[i]);
    if (c->evD[i]) cudaEventDestroy(c->evD[i]);
    if (c->evC[i]) cudaEventDestroy(c->evC[i]);
  }
  if (c->evFork) cudaEventDestroy(c->evFork);
  if (c->evJoinA) cudaEventDestroy(c->evJoinA);
  if (c->evJoinC) cudaEventDestroy(c->evJoinC);
  if (c->evJoinD) cudaEventDestroy(c->evJoinD);
  if (c->sU) cudaStreamDestroy(c->sU);
  if (c->sD) cudaStreamDestroy(c->sD);
  if (c->sP) cudaStreamDestroy(c->sP);
  for (int i = 0; i < 2; ++i)
    if (c->evP[i]) cudaEventDestroy(c->evP[i]);
  if (c->evJoinP) cudaEventDestroy(c->evJoinP);
  if (c->ex_phi) cudaFree(c->ex_phi);
  if (c->ex_V) cudaFree(c->ex_V);
  corr_ws_free(&c->corr_ws);
  for (auto& ev : c->corr_events) cudaEventDestroy(ev.first), cudaEventDestroy(ev.second);
  for (auto& ev : c->conv_events) cudaEventDestroy(ev.e0), cudaEventDestroy(ev.e1);
  delete c;
  return DVC_OK;
}

extern "C" const char* dvc_last_error(const dvc_ctx* c) { return c ? c->err.c_str() : g_create_err.c_str(); }

extern "C" int dvc_set_math(dvc_ctx* c, int conv_math, int corr_math) {
  if (!c) return DVC_ERR_ARG;
  if (conv_math != DVC_MATH_FP32 && conv_math != DVC_MATH_TF32X3) return fail(c, DVC_ERR_ARG, "conv math must be DVC_MATH_FP32 or DVC_MATH_TF32X3");
  if (conv_math != c->conv_math) c->ex_valid = false, c->warp_cache_valid = false;
  if (corr_math != DVC_MATH_FP32 && corr_math != DVC_MATH_TF32X3 && corr_math != DVC_MATH_BF16X3 && corr_math != DVC_MATH_FP16X3)
    return fail(c, DVC_ERR_ARG, "unknown corr math");
  c->conv_math = conv_math, c->corr_math = corr_math;
  return DVC_OK;
}

extern "C" int dvc_debug_set_flag(dvc_ctx* c, const char* name, int value) {
  if (!c || !name) return DVC_ERR_ARG;
  if (!strcmp(name, "two_level")) { c->two_level = value != 0; return DVC_OK; }
  if (!strcmp(name, "tc_kc")) { c->tc_kc = value < 1 ? 1 : value; return DVC_OK; }
  if (!strcmp(name, "corr_cluster")) { c->corr_cluster = value == 1 ? 1 : 2; return DVC_OK; }
  if (!strcmp(name, "corr_screen")) { c->corr_screen = value != 0; return DVC_OK; }
  if (!strcmp(name, "corr_phi_static")) {
    c->corr_phi_static = value != 0;
    c->corr_phi_key = c->corr_V_key = nullptr;  // the next call prepares the exemplar side afresh
    return DVC_OK;
  }
  if (!strcmp(name, "clip_astreams")) { c->clip_astreams = value == 2 ? 2 : 1; return DVC_OK; }
  if (!strcmp(name, "video_batch")) { c->video_batch = value < 1 ? 1 : (value > 64 ? 64 : value); return DVC_OK; }  // measurements
  if (!strcmp(name, "tc_tail")) { c->tc_tail = value < 0 ? 0 : value; return DVC_OK; }  // > 1: pretend pair-slot count (tests)
  if (!strcmp(name, "tc_f16")) { c->tc_f16 = value != 0; return DVC_OK; }
  if (!strcmp(name, "tc_splits")) { c->tc_splits = value < 0 ? 0 : (value > 8 ? 8 : value); return DVC_OK; }
  if (!strcmp(name, "tc_kbytes")) { c->tc_kbytes = value == 64 ? 64 : 128; return DVC_OK; }
  if (!strcmp(name, "tc_cluster")) { c->tc_cluster = value == 2 ? 2 : 1; return DVC_OK; }
  if (!strcmp(name, "tc_dbg")) { c->tc_dbg = value; return DVC_OK; }
  if (!strcmp(name, "tc_rowshare")) { c->tc_rowshare = value < 0 ? 0 : (value > 2 ? 2 : value); return DVC_OK; }
  if (!strcmp(name, "tc_force_bn")) {
    if (value != 0 && value != 64 && value != 128 && value != 256) return fail(c, DVC_ERR_ARG, "tc_force_bn must be 0, 64, 128 or 256");
    c->tc_force_bn = value;
    return DVC_OK;
  }
  return fail(c, DVC_ERR_ARG, std::string("unknown debug flag ") + name);
}

extern "C" int dvc_debug_get_buffer(dvc_ctx* c, const char* name, void** dev_ptr, int64_t* bytes, int* sig5) {
  if (!c || !name || !dev_ptr || !bytes) return DVC_ERR_ARG;
  if (!strcmp(name, "ex.phi")) { *dev_ptr = c->ex_phi; *bytes = (int64_t)c->ex_N * 256 * 4; return DVC_OK; }
  if (!strcmp(name, "ex.V")) { *dev_ptr = c->ex_V; *bytes = (int64_t)c->ex_N * 16; return DVC_OK; }
  auto it = c->bufs.find(name);
  if (it == c->bufs.end()) return fail(c, DVC_ERR_ARG, std::string("no such buffer: ") + name);
  *dev_ptr = it->second.p;
  *bytes = (int64_t)it->second.bytes;
  if (sig5) for (int i = 0; i < 5; ++i) sig5[i] = it->second.sig[i];
  return DVC_OK;
}

extern "C" int64_t dvc_launch_count(dvc_ctx*, int reset) {
  int64_t v = g_launches.load();
  if (reset) g_launches.store(0);
  return v;
}

extern "C" int dvc_profile_corr(dvc_ctx* c, int enable) {
  if (!c) return DVC_ERR_ARG;
  c->prof_corr = enable != 0;
  return DVC_OK;
}

extern "C" int dvc_profile_conv(dvc_ctx* c, int enable) {
  if (!c) return DVC_ERR_ARG;
  c->prof_conv = enable != 0;
  return DVC_OK;
}

// Sum of CUDA-event durations (ms) and of algorithmic FLOPs over the recorded tensor-core convolution launches of
// one kernel variant (64 / 128 / 256 = pixel-major channel tile, 1 = channel-major, 0 = all).  Returns launches.
extern "C" int dvc_conv_profile(dvc_ctx* c, int variant, int reset, double* total_ms, double* total_flops) {
  if (!c) return 0;
  double ms = 0.0, fl = 0.0;
  int n = 0;
  for (auto& ev : c->conv_events) {
    if (variant && ev.variant != variant) continue;
    if (cudaEventSynchronize(ev.e1) != cudaSuccess) continue;
    float t = 0.f;
    if (cudaEventElapsedTime(&t, ev.e0, ev.e1) == cudaSuccess) ms += t, fl += ev.flops, n++;
  }
  if (reset) {
    for (auto& ev : c->conv_events) cudaEventDestroy(ev.e0), cudaEventDestroy(ev.e1);
    c->conv_events.clear();
  }
  if (total_ms) *total_ms = ms;
  if (total_flops) *total_flops = fl;
  return n;
}

extern "C" double dvc_corr_mean_ms(dvc_ctx* c, int reset) {
  if (!c || c->corr_events.empty()) return 0.0;
  double tot = 0.0;
  int n = 0;
  for (auto& ev : c->corr_events) {
    if (cudaEventSynchronize(ev.second) != cudaSuccess) continue;
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, ev.first, ev.second) == cudaSuccess) tot += ms, n++;
  }
  if (reset) {
    for (auto& ev : c->corr_events) cudaEventDestroy(ev.first), cudaEventDestroy(ev.second);
    c->corr_events.clear();
  }
  return n ? tot / n : 0.0;
}

// ---- VGG19_pytorch.forward ----------------------------------------------------------------------
extern "C" int dvc_vgg19_forward(dvc_ctx* c, const float* x, int B, int H, int W, int preprocess, const char* const* keys,
                                 float* const* outs, int n_keys, void* stream) {
  if (!c || !x || !keys || !outs || B < 1 || n_keys < 1) return c ? fail(c, DVC_ERR_ARG, "vgg19_forward: bad argument") : DVC_ERR_ARG;
  if (H < 16 || W < 16) return fail(c, DVC_ERR_SHAPE, "vgg19_forward: H, W must be >= 16");
  cudaStream_t s = (cudaStream_t)stream;
  CUDA_TRY(c, cudaSetDevice(c->device));
  // deepest requested map decides where the trunk stops (the reference evaluates all 21 stages
  // regardless, NonlocalNet.py:235-255; the skipped tail is not observable)
  int deepest = -1;
  {
    int block = 1, idx = 1, pos = 0;
    for (const char* name : kVggSeq) {
      std::string key = name[0] == 'P' ? "p" + std::to_string(block) : "r" + std::to_string(block) + std::to_string(idx);
      if (name[0] == 'P') block++, idx = 1; else idx++;
      for (int i = 0; i < n_keys; ++i)
        if (keys[i] && key == keys[i] && pos > deepest) deepest = pos;
      pos++;
    }
  }
  std::string last_key;
  {
    int block = 1, idx = 1, pos = 0;
    for (const char* name : kVggSeq) {
      std::string key = name[0] == 'P' ? "p" + std::to_string(block) : "r" + std::to_string(block) + std::to_string(idx);
      if (name[0] == 'P') block++, idx = 1; else idx++;
      if (pos == deepest) last_key = key;
      pos++;
    }
  }
  if (deepest < 0) return fail(c, DVC_ERR_ARG, "vgg19_forward: unknown out_key");
  Act x0;
  DVC_TRY(stats_begin(c, s));
  DVC_TRY(get_act(c, "mvgg.x0", B, H, W, 8, 1, &x0, s));
  launch_nchw_to_act(x, 3, x0.d, nullptr, B, H, W, 8, 1, PAD_ZERO, preprocess ? 1 : 0, s);
  DVC_TRY(check_launch(c, "nchw_to_act"));
  VggMaps maps;
  DVC_TRY(vgg_trunk(c, "mvgg", x0, last_key, &maps, s));
  for (int i = 0; i < n_keys; ++i) {
    auto it = maps.m.find(keys[i] ? keys[i] : "");
    if (it == maps.m.end()) return fail(c, DVC_ERR_ARG, std::string("vgg19_forward: unknown out_key ") + (keys[i] ? keys[i] : "(null)"));
    const Act& a = it->second;
    if (a.h16)
      launch_act_to_nchw_h16(a.h16, a.l16, a.cell, a.H, a.W, a.P, a.C, a.C, outs[i], B, s);
    else
      launch_act_to_nchw(a.d, a.lo, a.H, a.W, a.P, a.C, 0, a.C, outs[i], B, s);
    DVC_TRY(check_launch(c, "act_to_nchw"));
  }
  return DVC_OK;
}

// ---- WarpNet.forward -----------------------------------------------------------------------------
static int features_from_nchw(dvc_ctx* c, const std::string& tag, const float* const* f, int B, int H, int W, Act n[4],
                              cudaStream_t s) {
  // dims the VGG trunk produces for an HxW input (floor-mode pools)
  const int hs[4] = {H / 2, H / 4, H / 8, H / 16}, ws[4] = {W / 2, W / 4, W / 8, W / 16}, cs[4] = {128, 256, 512, 512};
  for (int k = 0; k < 4; ++k) {
    DVC_TRY(get_act(c, tag + ".n" + std::to_string(k), B, hs[k], ws[k], cs[k], 1, &n[k], s, tc_mode(c)));
    launch_nchw_to_act(f[k], cs[k], n[k].d, n[k].lo, B, hs[k], ws[k], cs[k], 1, PAD_REFLECT, 0, s);
    DVC_TRY(check_launch(c, "nchw_to_act"));
  }
  return DVC_OK;
}

extern "C" int dvc_warpnet_forward(dvc_ctx* c, const float* B_lab_map, const float* const* A, const float* const* Bf, int B,
                                   int H, int W, float temperature, float wta, int reuse_exemplar, float* y, float* sim,
                                   void* stream) {
  if (!c || !B_lab_map || !A || !Bf || !y || !sim || B < 1) return c ? fail(c, DVC_ERR_ARG, "warpnet_forward: bad argument") : DVC_ERR_ARG;
  if (wta != 1.0f) return fail(c, DVC_ERR_ARG, "warpnet_forward: WTA_scale_weight != 1 is not supported (training-only path, NonlocalNet.py:486)");
  if (!(temperature > 0.f)) return fail(c, DVC_ERR_ARG, "warpnet_forward: temperature must be > 0");
  if (!legal_shape(H, W)) return fail(c, DVC_ERR_SHAPE, "warpnet_forward: H must be a multiple of 8 and W a multiple of 16 (the reference fails at NonlocalNet.py:464 otherwise)");
  cudaStream_t s = (cudaStream_t)stream;
  CUDA_TRY(c, cudaSetDevice(c->device));
  DVC_TRY(stats_begin(c, s));
  const int h = H / 4, w = W / 4, N = h * w;
  void *theta, *phi, *V, *yrows, *simrows;
  DVC_TRY(get_raw(c, "mwarp.theta", (size_t)B * N * 256 * 4, &theta, s));
  DVC_TRY(get_raw(c, "mwarp.phi", (size_t)B * N * 256 * 4, &phi, s));
  DVC_TRY(get_raw(c, "mwarp.V", (size_t)B * N * 4 * 4, &V, s));
  DVC_TRY(get_raw(c, "mwarp.yrows", (size_t)B * N * 4 * 4, &yrows, s));
  DVC_TRY(get_raw(c, "mwarp.simrows", (size_t)B * N * 4, &simrows, s));
  Act n[4];
  DVC_TRY(features_from_nchw(c, "mwarpA", A, B, H, W, n, s));
  DVC_TRY(warp_side(c, "mwarpA", n, "theta", (float*)theta, h, w, s));
  const bool can_reuse = reuse_exemplar && c->warp_cache_valid && c->warp_cache_sig[0] == B && c->warp_cache_sig[1] == H &&
                         c->warp_cache_sig[2] == W;
  if (!can_reuse) {
    DVC_TRY(features_from_nchw(c, "mwarpB", Bf, B, H, W, n, s));
    DVC_TRY(warp_side(c, "mwarpB", n, "phi", (float*)phi, h, w, s));
    launch_avgpool4_lab(B_lab_map, (float*)V, B, H, W, s);
    DVC_TRY(check_launch(c, "avgpool4"));
    c->warp_cache_valid = true;
    c->warp_cache_sig[0] = B, c->warp_cache_sig[1] = H, c->warp_cache_sig[2] = W;
  }
  CorrParams p{};
  p.theta = (float*)theta, p.phi = (float*)phi, p.V = (float*)V, p.B = B, p.Bphi = B, p.NA = N, p.NB = N, p.C = 256;
  p.temperature = temperature, p.y = (float*)yrows, p.sim = (float*)simrows, p.argmax = nullptr;
  DVC_TRY(run_corr(c, p, s));
  launch_rows_to_nchw_up4((float*)yrows, (float*)simrows, y, sim, B, h, w, s);
  return check_launch(c, "rows_to_nchw_up4");
}

// ---- ColorVidNet.forward -------------------------------------------------------------------------
extern "C" int dvc_colorvidnet_forward(dvc_ctx* c, const float* x, int B, int H, int W, float* out, void* stream) {
  if (!c || !x || !out || B < 1) return c ? fail(c, DVC_ERR_ARG, "colorvidnet_forward: bad argument") : DVC_ERR_ARG;
  if (H < 8 || W < 8 || H % 8 || W % 8) return fail(c, DVC_ERR_SHAPE, "colorvidnet_forward: H and W must be multiples of 8 (skip adds at ColorVidNet.py:129,135,140)");
  cudaStream_t s = (cudaStream_t)stream;
  CUDA_TRY(c, cudaSetDevice(c->device));
  DVC_TRY(stats_begin(c, s));
  Act in0;
  DVC_TRY(get_act(c, "mcolor.in0", B, H, W, 8, 1, &in0, s));
  launch_nchw_to_act(x, 7, in0.d, nullptr, B, H, W, 8, 1, PAD_ZERO, 0, s);
  DVC_TRY(check_launch(c, "nchw_to_act"));
  return colorvid(c, "mcolor", in0, out, s);
}

// ---- one convolution layer in isolation (test hook) ------------------------------------------------
// y = act(conv(pad(x)) + bias (+ add)) for the weights `name` of `net`, through exactly the engine, operand format and
// epilogue the layer programs use (tensor-core mode: fp16 planes with the static exponent of `in_bound`, or tf32 planes
// with tc_f16 = 0; CUDA-core mode otherwise).  out_planes = 1 stores the result as fp16 hi/lo planes with a
// device-derived exponent (the conv -> ReLU -> conv chains) and reads it back from them; upconv = 1 runs the four
// phase convolutions of a nearest-x2 + 3x3 decoder layer; fuse_tail = 1 the conv10_2 + conv10_ab + tanh epilogue
// (y is then [B][2][H][W]).  stats_out (device, [B][Cout][2] doubles) receives the InstanceNorm sums of the stored values.
extern "C" int dvc_debug_conv2d(dvc_ctx* c, int net, const char* name, const float* x, int B, int H, int W, int dil, int stride,
                                int act, float slope, int pad_mode, int upconv, int fuse_tail, float in_bound, int out_planes,
                                const float* add, float* y, double* stats_out, void* stream) {
  if (!c || !name || !x || !y || net < 0 || net > 2 || B < 1 || H < 1 || W < 1 || dil < 1 || (stride != 1 && stride != 2))
    return c ? fail(c, DVC_ERR_ARG, "debug_conv2d: bad argument") : DVC_ERR_ARG;
  cudaStream_t s = (cudaStream_t)stream;
  CUDA_TRY(c, cudaSetDevice(c->device));
  const ConvW* w;
  DVC_TRY(need_conv(c, net, name, &w));
  DVC_TRY(stats_begin(c, s));
  const bool tcm = tc_mode(c) && w->wt_hi, f16 = tcm && c->tc_f16;
  if ((upconv || fuse_tail) && !tcm) return fail(c, DVC_ERR_STATE, "debug_conv2d: phase / fused-tail layers need the tensor-core engine");
  if (out_planes && !f16) return fail(c, DVC_ERR_STATE, "debug_conv2d: device-scaled output planes need the fp16 engine");
  Act x0, xp, yo, addA;
  DVC_TRY(get_act(c, "dbg.x0", B, H, W, w->cin_pad, 0, &x0, s));
  launch_nchw_to_act(x, w->cin, x0.d, nullptr, B, H, W, w->cin_pad, 0, PAD_ZERO, 0, s);
  DVC_TRY(check_launch(c, "nchw_to_act"));
  DVC_TRY(get_act(c, "dbg.xp", B, H, W, w->cin_pad, w->k == 3 ? dil : 1, &xp, s, tcm ? (f16 ? 2 : 1) : 0));
  xp.e16 = e16_for(in_bound > 0.f ? in_bound : 1.0);
  XfOpt xo;
  xo.pad_mode = pad_mode ? PAD_REFLECT : PAD_ZERO;
  DVC_TRY(run_xform(c, x0, xp, xo, s));
  const int Ho = upconv ? 2 * H : (H + stride - 1) / stride, Wo = upconv ? 2 * W : (W + stride - 1) / stride;
  ConvOpt o;
  o.dil = dil, o.stride = stride, o.act = act, o.slope = slope;
  if (add) {
    DVC_TRY(get_act(c, "dbg.add", B, Ho, Wo, w->cout_pad, 0, &addA, s));
    launch_nchw_to_act(add, w->cout, addA.d, nullptr, B, Ho, Wo, w->cout_pad, 0, PAD_ZERO, 0, s);
    DVC_TRY(check_launch(c, "nchw_to_act"));
    if (out_planes) {
      DVC_TRY(cell_alloc(c, &addA.cell, s));
      launch_amax(addA.d, addA.elems(), addA.cell, s);
      DVC_TRY(check_launch(c, "amax"));
    }
    o.add = &addA;
  }
  double* st = nullptr;
  if (stats_out) {
    DVC_TRY(stats_alloc(c, B, w->cout, &st, s));
    o.stats = st;
  }
  if (fuse_tail) {
    const float *wab, *bab;
    DVC_TRY(need_vec(c, DVC_NET_COLOR, "conv10_ab", &wab));
    DVC_TRY(need_vec(c, DVC_NET_COLOR, "conv10_ab.bias", &bab));
    if (w->cout != 128) return fail(c, DVC_ERR_SHAPE, "debug_conv2d: the fused tail needs 128 output channels");
    yo.B = B, yo.H = Ho, yo.W = Wo, yo.C = w->cout, yo.P = 0;
    o.fin_w = wab, o.fin_b = bab, o.fin_out = y;
    return run_conv(c, w, xp, yo, o, s);
  }
  DVC_TRY(get_act(c, "dbg.y", B, Ho, Wo, w->cout, out_planes ? 1 : 0, &yo, s, out_planes ? 2 : 0));
  if (out_planes) DVC_TRY(cell_alloc(c, &yo.cell, s));
  if (upconv) {
    float l1 = 0.f;
    for (int ph = 0; ph < 4; ++ph) {
      auto it = c->conv[net].find(std::string(name) + "#p" + std::to_string(ph));
      if (it == c->conv[net].end() || !it->second.w16_hi) return fail(c, DVC_ERR_STATE, std::string("phase weights missing: ") + name);
      l1 = fmaxf(l1, it->second.l1max);
    }
    for (int ph = 0; ph < 4; ++ph) {
      ConvW pw = c->conv[net][std::string(name) + "#p" + std::to_string(ph)];
      pw.b = w->b, pw.bmax = w->bmax;
      ConvOpt op = o;
      op.phase = ph, op.l1_override = l1;
      DVC_TRY(run_conv(c, &pw, xp, yo, op, s));
    }
  } else {
    DVC_TRY(run_conv(c, w, xp, yo, o, s));
  }
  if (yo.h16)
    launch_act_to_nchw_h16(yo.h16, yo.l16, yo.cell, yo.H, yo.W, yo.P, yo.C, w->cout, y, B, s);
  else
    launch_act_to_nchw(yo.d, yo.lo, yo.H, yo.W, yo.P, yo.C, 0, w->cout, y, B, s);
  DVC_TRY(check_launch(c, "act_to_nchw"));
  if (stats_out) CUDA_TRY(c, cudaMemcpyAsync(stats_out, st, (size_t)B * w->cout * 2 * sizeof(double), cudaMemcpyDeviceToDevice, s));
  return DVC_OK;
}

// ---- stand-alone correlation ---------------------------------------------------------------------
extern "C" int dvc_corr_softmax_warp(dvc_ctx* c, const float* theta_hat, const float* phi_hat, const float* V, int B,
                                     int Bphi, int NA, int NB, int C, float temperature, float* y, float* sim,
                                     int32_t* argmax, void* stream) {
  if (!c || !theta_hat || !phi_hat || !V || !y || !sim) return c ? fail(c, DVC_ERR_ARG, "corr: bad argument") : DVC_ERR_ARG;
  if (C < 64 || C % 64 || C > 4096) return fail(c, DVC_ERR_SHAPE, "corr: C must be a multiple of 64 (WarpNet.inter_channels is 256)");
  if (C != 256 && c->corr_math == DVC_MATH_FP32) return fail(c, DVC_ERR_SHAPE, "corr: the CUDA-core twin is built for C = 256");
  if (B < 1 || NA < 1 || NB < 1 || (Bphi != B && Bphi != 1)) return fail(c, DVC_ERR_SHAPE, "corr: bad sizes");
  if (!(temperature > 0.f)) return fail(c, DVC_ERR_ARG, "corr: temperature must be > 0");
  cudaStream_t s = (cudaStream_t)stream;
  CUDA_TRY(c, cudaSetDevice(c->device));
  void *th, *ph, *V4, *y4;
  DVC_TRY(get_raw(c, "corr.theta", (size_t)B * NA * C * 4, &th, s));
  DVC_TRY(get_raw(c, "corr.phi", (size_t)Bphi * NB * C * 4, &ph, s));
  DVC_TRY(get_raw(c, "corr.V4", (size_t)Bphi * NB * 16, &V4, s));
  DVC_TRY(get_raw(c, "corr.y4", (size_t)B * NA * 16, &y4, s));
  // channel-major [b][C][N] (the reference's view, NonlocalNet.py:468,473) -> position-major rows
  launch_transpose_cn(theta_hat, (float*)th, B, C, NA, s);
  const long long dims = ((long long)Bphi << 40) ^ ((long long)NB << 8) ^ C;
  const bool phi_ready = c->corr_phi_static && c->corr_phi_key == phi_hat && c->corr_V_key == V && c->corr_phi_dims == dims;
  if (!phi_ready) {
    launch_transpose_cn(phi_hat, (float*)ph, Bphi, C, NB, s);
    // rows (L, a, b, 1): the 4th lane is the constant the softmax epilogue sums the weights with
    launch_pack_v4(V, (float*)V4, (size_t)Bphi * NB, s);
    DVC_TRY(check_launch(c, "pack_v4"));
    c->corr_phi_key = phi_hat, c->corr_V_key = V, c->corr_phi_dims = dims, c->corr_phi_version++;
  }
  CorrParams p{};
  p.theta = (float*)th, p.phi = (float*)ph, p.V = (float*)V4, p.B = B, p.Bphi = Bphi, p.NA = NA, p.NB = NB, p.C = C;
  p.temperature = temperature, p.y = (float*)y4, p.sim = sim, p.argmax = argmax;
  if (c->corr_peers.n > 0) {
    if (B != 1) return fail(c, DVC_ERR_SHAPE, "corr: peer outputs need B = 1");
    if (c->corr_math == DVC_MATH_FP32) return fail(c, DVC_ERR_STATE, "corr: peer outputs need a tensor-core correlation mode");
    p.peers = c->corr_peers;
  }
  // a version number lets the correlation keep the exemplar's operand planes too (offset: never collides with ex_version)
  DVC_TRY(run_corr(c, p, s, c->corr_phi_static ? (1ll << 40) + c->corr_phi_version : -1));
  CUDA_TRY(c, cudaMemcpy2DAsync(y, 12, y4, 16, 12, (size_t)B * NA, cudaMemcpyDeviceToDevice, s));
  return DVC_OK;
}

// ---- query-row-sharded correlation: peer-mapped result buffers (CUDA IPC between the per-GPU processes) -----------
extern "C" int dvc_peer_buffer_create(dvc_ctx* c, int64_t bytes, void** dev_ptr, unsigned char* handle64) {
  if (!c || !dev_ptr || !handle64 || bytes < 1) return c ? fail(c, DVC_ERR_ARG, "peer_buffer_create: bad argument") : DVC_ERR_ARG;
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
  CUDA_TRY(c, cudaSetDevice(c->device));
  void* p = nullptr;
  CUDA_TRY(c, cudaMalloc(&p, (size_t)bytes));
  CUDA_TRY(c, cudaMemset(p, 0, (size_t)bytes));
  cudaIpcMemHandle_t h;
  cudaError_t e = cudaIpcGetMemHandle(&h, p);
  if (e != cudaSuccess) {
    cudaFree(p);
    return fail(c, DVC_ERR_CUDA, std::string("cudaIpcGetMemHandle: ") + cudaGetErrorString(e));
  }
  memcpy(handle64, &h, 64);
  *dev_ptr = p;
  return DVC_OK;
}

extern "C" int dvc_peer_buffer_open(dvc_ctx* c, const unsigned char* handle64, void** dev_ptr) {
  if (!c || !dev_ptr || !handle64) return c ? fail(c, DVC_ERR_ARG, "peer_buffer_open: bad argument") : DVC_ERR_ARG;
  CUDA_TRY(c, cudaSetDevice(c->device));
  cudaIpcMemHandle_t h;
  memcpy(&h, handle64, 64);
  void* p = nullptr;
  CUDA_TRY(c, cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
  *dev_ptr = p;
  return DVC_OK;
}

extern "C" int dvc_peer_buffer_close(dvc_ctx* c, void* opened_ptr) {
  if (!c || !opened_ptr) return c ? fail(c, DVC_ERR_ARG, "peer_buffer_close: bad argument") : DVC_ERR_ARG;
  CUDA_TRY(c, cudaSetDevice(c->device));
  CUDA_TRY(c, cudaIpcCloseMemHandle(opened_ptr));
  return DVC_OK;
}

extern "C" int dvc_peer_buffer_destroy(dvc_ctx* c, void* created_ptr) {
  if (!c || !created_ptr) return c ? fail(c, DVC_ERR_ARG, "peer_buffer_destroy: bad argument") : DVC_ERR_ARG;
  CUDA_TRY(c, cudaSetDevice(c->device));
  CUDA_TRY(c, cudaFree(created_ptr));
  return DVC_OK;
}

extern "C" int dvc_corr_set_peer_outputs(dvc_ctx* c, int n, float* const* y4, float* const* sim, int64_t row0) {
  if (!c || n < 0 || n > 8 || row0 < 0 || (n > 0 && (!y4 || !sim))) return c ? fail(c, DVC_ERR_ARG, "corr_set_peer_outputs: bad argument") : DVC_ERR_ARG;
  c->corr_peers = CorrPeers();
  for (int g = 0; g < n; ++g) {
    if (!y4[g] || !sim[g]) return fail(c, DVC_ERR_ARG, "corr_set_peer_outputs: null destination");
    c->corr_peers.y4[g] = y4[g], c->corr_peers.sim[g] = sim[g];
  }
  c->corr_peers.n = n, c->corr_peers.row0 = row0;
  return DVC_OK;
}

// ---- fused per-frame path ---------------------------------------------------------------------------
static int normalised_features(dvc_ctx* c, const std::string& tag, VggMaps& maps, Act n[4], cudaStream_t s) {
  const char* keys[4] = {"r22", "r32", "r42", "r52"};
  for (int k = 0; k < 4; ++k) {
    const Act& r = maps.m[keys[k]];
    // unit-L2 pixels: |x| <= 1, fp16 planes of x * 2^14
    DVC_TRY(get_act(c, tag + ".n" + std::to_string(k), r.B, r.H, r.W, r.C, 1, &n[k], s, tc_mode(c) ? (c->tc_f16 ? 2 : 1) : 0));
    n[k].e16 = 14;
    DVC_TRY(run_pixnorm(c, r, n[k].d, n[k].lo, 1, PAD_REFLECT, nullptr, 1.0, s, n[k].h16, n[k].l16, n[k].e16));  // feature_normalize, util.py:155-158
  }
  return DVC_OK;
}

extern "C" int dvc_set_exemplar(dvc_ctx* c, const float* IB_lab, int H, int W, void* stream) {
  if (!c || !IB_lab) return c ? fail(c, DVC_ERR_ARG, "set_exemplar: bad argument") : DVC_ERR_ARG;
  if (!legal_shape(H, W)) return fail(c, DVC_ERR_SHAPE, "set_exemplar: H must be a multiple of 8 and W a multiple of 16");
  cudaStream_t s = (cudaStream_t)stream;
  CUDA_TRY(c, cudaSetDevice(c->device));
  DVC_TRY(stats_begin(c, s));
  void* lab;
  DVC_TRY(get_raw(c, "ex.lab", (size_t)3 * H * W * 4, &lab, s));
  CUDA_TRY(c, cudaMemcpyAsync(lab, IB_lab, (size_t)3 * H * W * 4, cudaMemcpyDefault, s));
  Act x0;
  DVC_TRY(get_act(c, "ex.x0", 1, H, W, 8, 1, &x0, s));
  launch_nchw_to_act((float*)lab, 3, x0.d, nullptr, 1, H, W, 8, 1, PAD_ZERO, 3, s);  // test.py:61-65
  DVC_TRY(check_launch(c, "nchw_to_act"));
  VggMaps maps;
  DVC_TRY(vgg_trunk(c, "ex", x0, "r52", &maps, s));
  Act n[4];
  DVC_TRY(normalised_features(c, "ex", maps, n, s));
  const int h = H / 4, w = W / 4, N = h * w;
  if (c->ex_N != N) {
    if (c->ex_phi) cudaFree(c->ex_phi);
    if (c->ex_V) cudaFree(c->ex_V);
    c->ex_phi = c->ex_V = nullptr;
    CUDA_TRY(c, cudaMalloc((void**)&c->ex_phi, (size_t)N * 256 * 4));
    CUDA_TRY(c, cudaMalloc((void**)&c->ex_V, (size_t)N * 16));
    c->ex_N = N;
  }
  DVC_TRY(warp_side(c, "ex", n, "phi", c->ex_phi, h, w, s));
  launch_avgpool4_lab((float*)lab, c->ex_V, 1, H, W, s);
  DVC_TRY(check_launch(c, "avgpool4"));
  c->ex_H = H, c->ex_W = W, c->ex_valid = true, c->ex_version++;
  // the frame loop must not allocate: size the correlation workspace for one frame against this exemplar now
  if (corr_ws_reserve(&c->corr_ws, 1, 1, N, N) != 0) return fail(c, DVC_ERR_CUDA, "set_exemplar: correlation workspace allocation failed");
  return DVC_OK;
}

// Phase A (independent of the previous frame): VGG19 -> feature_normalize -> WarpNet A side -> correlation.
static int frames_phaseA(dvc_ctx* c, const std::string& tag, const float* IA_l, int B, int H, int W, float temperature,
                         float* yrows, float* simrows, cudaStream_t s, int arena = 0, CorrWorkspace* ws = nullptr) {
  DVC_TRY(stats_begin(c, s, arena));
  const int h = H / 4, w = W / 4, N = h * w;
  Act x0;
  DVC_TRY(get_act(c, tag + ".x0", B, H, W, 8, 1, &x0, s));
  launch_nchw_to_act(IA_l, 1, x0.d, nullptr, B, H, W, 8, 1, PAD_ZERO, 2, s);  // FrameColor.py:6 + util.py:347-352
  DVC_TRY(check_launch(c, "nchw_to_act"));
  VggMaps maps;
  DVC_TRY(vgg_trunk(c, tag, x0, "r52", &maps, s));
  Act n[4];
  DVC_TRY(normalised_features(c, tag, maps, n, s));
  void* theta;
  DVC_TRY(get_raw(c, tag + ".theta", (size_t)B * N * 256 * 4, &theta, s));
  DVC_TRY(warp_side(c, tag, n, "theta", (float*)theta, h, w, s));
  CorrParams p{};
  p.theta = (float*)theta, p.phi = c->ex_phi, p.V = c->ex_V, p.B = B, p.Bphi = 1, p.NA = N, p.NB = N, p.C = 256;
  p.temperature = temperature, p.y = yrows, p.sim = simrows, p.argmax = nullptr;
  return run_corr(c, p, s, c->ex_version, ws);
}

// Phase C (the recurrent part): ColorVidNet on [L, warped ab, similarity, previous Lab] (FrameColor.py:63-65).
static int frames_phaseC(dvc_ctx* c, const std::string& tag, const float* IA_l, const float* yrows, const float* simrows,
                         const float* IA_last_lab, int B, int H, int W, float* out_ab, cudaStream_t s) {
  DVC_TRY(stats_begin(c, s, 1));
  Act in0;
  DVC_TRY(get_act(c, tag + ".in0", B, H, W, 8, 1, &in0, s));
  launch_build_color_input(IA_l, yrows, simrows, IA_last_lab, in0.d, B, H, W, 1, s);
  DVC_TRY(check_launch(c, "build_color_input"));
  return colorvid(c, tag, in0, out_ab, s);
}

static int check_frame_args(dvc_ctx* c, int H, int W, float temperature) {
  if (!c->ex_valid) return fail(c, DVC_ERR_STATE, "colorize: call dvc_set_exemplar first");
  if (H != c->ex_H || W != c->ex_W) return fail(c, DVC_ERR_SHAPE, "colorize: frame size differs from the exemplar's");
  if (!(temperature > 0.f)) return fail(c, DVC_ERR_ARG, "colorize: temperature must be > 0");
  return DVC_OK;
}

extern "C" int dvc_colorize_frames(dvc_ctx* c, const float* IA_l, const float* IA_last_lab, int B, int H, int W,
                                   float temperature, float* out_ab, float* out_warp_lab, float* out_sim, void* stream) {
  if (!c || !IA_l || !IA_last_lab || !out_ab || B < 1) return c ? fail(c, DVC_ERR_ARG, "colorize_frames: bad argument") : DVC_ERR_ARG;
  DVC_TRY(check_frame_args(c, H, W, temperature));
  cudaStream_t s = (cudaStream_t)stream;
  CUDA_TRY(c, cudaSetDevice(c->device));
  const int h = H / 4, w = W / 4, N = h * w;
  void *yrows, *simrows;
  DVC_TRY(get_raw(c, "fr.yrows", (size_t)B * N * 16, &yrows, s));
  DVC_TRY(get_raw(c, "fr.simrows", (size_t)B * N * 4, &simrows, s));
  DVC_TRY(frames_phaseA(c, "fr", IA_l, B, H, W, temperature, (float*)yrows, (float*)simrows, s));
  if (out_warp_lab || out_sim) {
    launch_rows_to_nchw_up4((float*)yrows, (float*)simrows, out_warp_lab, out_sim, B, h, w, s);
    DVC_TRY(check_launch(c, "rows_to_nchw_up4"));
  }
  return frames_phaseC(c, "fr", IA_l, (float*)yrows, (float*)simrows, IA_last_lab, B, H, W, out_ab, s);
}

static int clip_streams(dvc_ctx* c) {
  if (c->sA) return DVC_OK;
  CUDA_TRY(c, cudaStreamCreateWithFlags(&c->sA, cudaStreamNonBlocking));
  CUDA_TRY(c, cudaStreamCreateWithFlags(&c->sA2, cudaStreamNonBlocking));
  CUDA_TRY(c, cudaEventCreateWithFlags(&c->evJoinA2, cudaEventDisableTiming));
  CUDA_TRY(c, cudaStreamCreateWithFlags(&c->sC, cudaStreamNonBlocking));
  CUDA_TRY(c, cudaStreamCreateWithFlags(&c->sU, cudaStreamNonBlocking));
  CUDA_TRY(c, cudaStreamCreateWithFlags(&c->sD, cudaStreamNonBlocking));
  CUDA_TRY(c, cudaEventCreateWithFlags(&c->evJoinD, cudaEventDisableTiming));
  for (int i = 0; i < 4; ++i) {
    CUDA_TRY(c, cudaEventCreateWithFlags(&c->evU[i], cudaEventDisableTiming));
    CUDA_TRY(c, cudaEventCreateWithFlags(&c->evD[i], cudaEventDisableTiming));
    CUDA_TRY(c, cudaEventCreateWithFlags(&c->evA[i], cudaEventDisableTiming));
    CUDA_TRY(c, cudaEventCreateWithFlags(&c->evC[i], cudaEventDisableTiming));
  }
  CUDA_TRY(c, cudaEventCreateWithFlags(&c->evFork, cudaEventDisableTiming));
  CUDA_TRY(c, cudaEventCreateWithFlags(&c->evJoinA, cudaEventDisableTiming));
  CUDA_TRY(c, cudaEventCreateWithFlags(&c->evJoinC, cudaEventDisableTiming));
  CUDA_TRY(c, cudaStreamCreateWithFlags(&c->sP, cudaStreamNonBlocking));
  CUDA_TRY(c, cudaEventCreateWithFlags(&c->evP[0], cudaEventDisableTiming));
  CUDA_TRY(c, cudaEventCreateWithFlags(&c->evP[1], cudaEventDisableTiming));
  CUDA_TRY(c, cudaEventCreateWithFlags(&c->evJoinP, cudaEventDisableTiming));
  return DVC_OK;
}

// Per-frame stages of the clip driver around the two network phases (dvc_colorize_clip: plain copies of L and ab;
// dvc_colorize_video_rgb8: uint8 frames in, ingest, batched post-processing, uint8 frames out).
struct ClipStages {
  // upload stream: frame t's half-size L into the slot Lt (the driver has made su wait until the slot is free)
  std::function<int(int t, float* Lt, cudaStream_t su)> ingest;
  // the half-size ab slot frame t's ColorVidNet writes; makes sc wait until the slot is free
  std::function<int(int t, cudaStream_t sc, float** abt)> ab_slot;
  // hands frame t's ab on once `done` (recorded on the ColorVidNet stream after frame t) has fired
  std::function<int(int t, const float* abt, cudaEvent_t done)> egress;
};

// test.py:68-96 for one contiguous segment of F frames, starting from the previous frame's Lab in `dlast` (updated in place).
// Frame t+1's frame-independent phase (VGG / WarpNet / correlation) runs on stream A while frame t's ColorVidNet -- which
// needs frame t-1's prediction -- runs on stream C; the partial waves of either leave SMs idle that the other fills.
// Ingest (up to four frames ahead) and egress run on their own streams so that neither compute stream waits for PCIe.
static int run_clip(dvc_ctx* c, int F, int H, int W, float temperature, float* dlast, const ClipStages& st, cudaStream_t s) {
  const size_t hw = (size_t)H * W;
  const int N = (H / 4) * (W / 4);
  void *dL, *yrows, *simrows;
  DVC_TRY(get_raw(c, "clip.L", 4 * hw * 4, &dL, s));   // 4 slots
  DVC_TRY(get_raw(c, "clip.yrows", (size_t)4 * N * 16, &yrows, s));  // 4 slots: phase A may run up to 3 frames ahead
  DVC_TRY(get_raw(c, "clip.simrows", (size_t)4 * N * 4, &simrows, s));
  const bool two_a = c->clip_astreams == 2;
  // the second phase-A stream has its own correlation workspace (sized like the first at dvc_set_exemplar time)
  if (two_a && corr_ws_reserve(&c->corr_ws2, 1, 1, N, N) != 0) return fail(c, DVC_ERR_CUDA, "colorize_clip: correlation workspace allocation failed");
  // Every exit below goes through the join epilogue: an error in the middle of the loop must not return while copies
  // or kernels of earlier frames are still writing into the outputs / the slots (a retry would race with them).
  auto enqueue = [&]() -> int {
    CUDA_TRY(c, cudaEventRecord(c->evFork, s));
    for (cudaStream_t si : {c->sA, c->sA2, c->sC, c->sU, c->sD, c->sP}) CUDA_TRY(c, cudaStreamWaitEvent(si, c->evFork, 0));
    for (int t = 0; t < F; ++t) {
      float* Lt = (float*)dL + (size_t)(t & 3) * hw;
      float* yr = (float*)yrows + (size_t)(t & 3) * N * 4;
      float* sr = (float*)simrows + (size_t)(t & 3) * N;
      const bool odd = two_a && (t & 1);
      cudaStream_t sAt = odd ? c->sA2 : c->sA;
      // ---- upload stream: the L slot was last read by frame t-4's ColorVidNet / make_last ----
      if (t >= 4) CUDA_TRY(c, cudaStreamWaitEvent(c->sU, c->evC[(t - 4) & 3], 0));
      DVC_TRY(st.ingest(t, Lt, c->sU));
      CUDA_TRY(c, cudaEventRecord(c->evU[t & 3], c->sU));
      // ---- stream A (two of them, alternating, when clip_astreams = 2): the frame-independent phase; the reuse of the
      // warp-row slot waits for frame t-4's ColorVidNet ----
      CUDA_TRY(c, cudaStreamWaitEvent(sAt, c->evU[t & 3], 0));
      if (t >= 4) CUDA_TRY(c, cudaStreamWaitEvent(sAt, c->evC[(t - 4) & 3], 0));
      DVC_TRY(frames_phaseA(c, odd ? "clipA2" : "clipA", Lt, 1, H, W, temperature, yr, sr, sAt, odd ? 2 : 0, odd ? &c->corr_ws2 : nullptr));
      CUDA_TRY(c, cudaEventRecord(c->evA[t & 3], sAt));
      // ---- stream C: the recurrent phase ----
      CUDA_TRY(c, cudaStreamWaitEvent(c->sC, c->evA[t & 3], 0));
      float* abt = nullptr;
      DVC_TRY(st.ab_slot(t, c->sC, &abt));
      DVC_TRY(frames_phaseC(c, "clipC", Lt, yr, sr, dlast, 1, H, W, abt, c->sC));
      launch_make_last(Lt, abt, dlast, 1, H, W, c->sC);  // test.py:96
      DVC_TRY(check_launch(c, "make_last"));
      CUDA_TRY(c, cudaEventRecord(c->evC[t & 3], c->sC));
      DVC_TRY(st.egress(t, abt, c->evC[t & 3]));
    }
    return DVC_OK;
  };
  const int rc = enqueue();
  const std::string first_err = c->err;
  // join: the caller's stream waits for the internal streams, then the host waits for the caller's stream
  bool join_ok = true;
  join_ok &= cudaEventRecord(c->evJoinA, c->sA) == cudaSuccess && cudaStreamWaitEvent(s, c->evJoinA, 0) == cudaSuccess;
  join_ok &= cudaEventRecord(c->evJoinA2, c->sA2) == cudaSuccess && cudaStreamWaitEvent(s, c->evJoinA2, 0) == cudaSuccess;
  join_ok &= cudaEventRecord(c->evJoinC, c->sC) == cudaSuccess && cudaStreamWaitEvent(s, c->evJoinC, 0) == cudaSuccess;
  join_ok &= cudaEventRecord(c->evJoinD, c->sD) == cudaSuccess && cudaStreamWaitEvent(s, c->evJoinD, 0) == cudaSuccess;
  join_ok &= cudaEventRecord(c->evJoinP, c->sP) == cudaSuccess && cudaStreamWaitEvent(s, c->evJoinP, 0) == cudaSuccess;
  join_ok &= cudaEventRecord(c->evFork, c->sU) == cudaSuccess && cudaStreamWaitEvent(s, c->evFork, 0) == cudaSuccess;
  const cudaError_t se = cudaStreamSynchronize(s);
  if (rc != DVC_OK) {
    if (!join_ok || se != cudaSuccess) {  // could not even drain the streams: make sure nothing is in flight
      for (cudaStream_t si : {c->sA, c->sA2, c->sC, c->sU, c->sD, c->sP}) cudaStreamSynchronize(si);
    }
    c->err = first_err;
    return rc;
  }
  if (!join_ok) return fail(c, DVC_ERR_CUDA, "colorize_clip: joining the internal streams failed");
  if (se != cudaSuccess) return fail(c, DVC_ERR_CUDA, std::string("colorize_clip: ") + cudaGetErrorString(se));
  return DVC_OK;
}

// L / ab may be host (pinned) or device memory.
extern "C" int dvc_colorize_clip(dvc_ctx* c, const float* L_in, int F, int H, int W, float temperature,
                                 const float* first_last, float* ab_out, void* stream) {
  if (!c || !L_in || !ab_out || F < 1) return c ? fail(c, DVC_ERR_ARG, "colorize_clip: bad argument") : DVC_ERR_ARG;
  DVC_TRY(check_frame_args(c, H, W, temperature));
  cudaStream_t s = (cudaStream_t)stream;
  CUDA_TRY(c, cudaSetDevice(c->device));
  DVC_TRY(clip_streams(c));
  const size_t hw = (size_t)H * W;
  void *dlast, *dab;
  DVC_TRY(get_raw(c, "clip.last", 3 * hw * 4, &dlast, s));
  DVC_TRY(get_raw(c, "clip.ab", 2 * 2 * hw * 4, &dab, s));  // 2 slots
  if (first_last)
    CUDA_TRY(c, cudaMemcpyAsync(dlast, first_last, 3 * hw * 4, cudaMemcpyDefault, s));
  else
    CUDA_TRY(c, cudaMemsetAsync(dlast, 0, 3 * hw * 4, s));  // test.py:80
  ClipStages st;
  st.ingest = [&](int t, float* Lt, cudaStream_t su) -> int {
    CUDA_TRY(c, cudaMemcpyAsync(Lt, L_in + (size_t)t * hw, hw * 4, cudaMemcpyDefault, su));
    return DVC_OK;
  };
  st.ab_slot = [&](int t, cudaStream_t sc, float** abt) -> int {
    if (t >= 2) CUDA_TRY(c, cudaStreamWaitEvent(sc, c->evD[(t - 2) & 3], 0));  // the ab slot has been downloaded
    *abt = (float*)dab + (size_t)(t & 1) * 2 * hw;
    return DVC_OK;
  };
  st.egress = [&](int t, const float* abt, cudaEvent_t done) -> int {
    CUDA_TRY(c, cudaStreamWaitEvent(c->sD, done, 0));
    CUDA_TRY(c, cudaMemcpyAsync(ab_out + (size_t)t * 2 * hw, abt, 2 * hw * 4, cudaMemcpyDefault, c->sD));
    CUDA_TRY(c, cudaEventRecord(c->evD[t & 3], c->sD));
    return DVC_OK;
  };
  return run_clip(c, F, H, W, temperature, (float*)dlast, st, s);
}

// ---- pre / post-processing around the nets (SURVEY.md §8f row 1) -----------------------------------------
extern "C" int dvc_resize_half(dvc_ctx* c, const float* dev_src, int planes, int H, int W, float* dev_dst, void* stream) {
  if (!c || !dev_src || !dev_dst || planes < 1) return c ? fail(c, DVC_ERR_ARG, "resize_half: bad argument") : DVC_ERR_ARG;
  if (H < 2 || W < 2 || (H & 1) || (W & 1)) return fail(c, DVC_ERR_SHAPE, "resize_half: H and W must be even");
  CUDA_TRY(c, cudaSetDevice(c->device));
  launch_resize_half(dev_src, dev_dst, planes, H, W, (cudaStream_t)stream);
  return check_launch(c, "resize_half");
}

extern "C" int dvc_upsample2_scaled(dvc_ctx* c, const float* dev_src, int planes, int h, int w, float scale, float* dev_dst,
                                    void* stream) {
  if (!c || !dev_src || !dev_dst || planes < 1 || h < 1 || w < 1) return c ? fail(c, DVC_ERR_ARG, "upsample2: bad argument") : DVC_ERR_ARG;
  CUDA_TRY(c, cudaSetDevice(c->device));
  launch_upsample2(dev_src, dev_dst, planes, h, w, scale, (cudaStream_t)stream);
  return check_launch(c, "upsample2");
}

// rgb_from_xyz = inv(xyz_from_rgb) (skimage.color.colorconv), by the adjugate in double precision
static void rgb_from_xyz(double inv[9]) {
  const double a[9] = {0.412453, 0.357580, 0.180423, 0.212671, 0.715160, 0.072169, 0.019334, 0.119193, 0.950227};
  const double det = a[0] * (a[4] * a[8] - a[5] * a[7]) - a[1] * (a[3] * a[8] - a[5] * a[6]) + a[2] * (a[3] * a[7] - a[4] * a[6]);
  const double m[9] = {(a[4] * a[8] - a[5] * a[7]) / det, (a[2] * a[7] - a[1] * a[8]) / det, (a[1] * a[5] - a[2] * a[4]) / det,
                       (a[5] * a[6] - a[3] * a[8]) / det, (a[0] * a[8] - a[2] * a[6]) / det, (a[2] * a[3] - a[0] * a[5]) / det,
                       (a[3] * a[7] - a[4] * a[6]) / det, (a[1] * a[6] - a[0] * a[7]) / det, (a[0] * a[4] - a[1] * a[3]) / det};
  for (int i = 0; i < 9; ++i) inv[i] = m[i];
}

extern "C" int dvc_lab_to_rgb8(dvc_ctx* c, const float* dev_l, const float* dev_ab, int B, int H, int W, unsigned char* dev_rgb,
                               void* stream) {
  if (!c || !dev_l || !dev_ab || !dev_rgb || B < 1 || H < 1 || W < 1) return c ? fail(c, DVC_ERR_ARG, "lab_to_rgb8: bad argument") : DVC_ERR_ARG;
  CUDA_TRY(c, cudaSetDevice(c->device));
  double inv[9];
  rgb_from_xyz(inv);
  launch_lab_to_rgb8(dev_l, dev_ab, dev_rgb, B, H, W, inv, (cudaStream_t)stream);
  return check_launch(c, "lab_to_rgb8");
}

extern "C" int dvc_rgb8_to_lab(dvc_ctx* c, const unsigned char* dev_rgb, int B, int H, int W, float* dev_lab, void* stream) {
  if (!c || !dev_rgb || !dev_lab || B < 1 || H < 1 || W < 1) return c ? fail(c, DVC_ERR_ARG, "rgb8_to_lab: bad argument") : DVC_ERR_ARG;
  CUDA_TRY(c, cudaSetDevice(c->device));
  launch_rgb8_to_lab(dev_rgb, dev_lab, B, H, W, (cudaStream_t)stream);
  return check_launch(c, "rgb8_to_lab");
}

// ---- ContextualLoss_forward (models/ContextualLoss.py:82-126; train.py's default "forward" direction), forward value only --
// CX_b = mean_i max_j A_ij, A_ij = w_ij / sum_j w_ij, w_ij = exp((1 - d_ij / (min_j d_ij + 1e-5)) / h), d = 1 - X^T Y on centred,
// unit-norm feature columns.  With m_i = max_j f_ij (f = X^T Y): max_j A_ij = 1 / sum_j exp((f_ij - m_i) / T_i),
// T_i = h (1 - m_i + 1e-5) -- the row maximum (first pass of K7) and then K7's online softmax with a per-row temperature.
extern "C" int dvc_contextual_loss_forward(dvc_ctx* c, const float* dev_X, const float* dev_Y, int B, int C, int NX, int NY, float h,
                                           int feature_centering, float* dev_loss, void* stream) {
  if (!c || !dev_X || !dev_Y || !dev_loss || B < 1 || NX < 1 || NY < 1) return c ? fail(c, DVC_ERR_ARG, "contextual_loss: bad argument") : DVC_ERR_ARG;
  if (C < 64 || C % 64 || C > 4096) return fail(c, DVC_ERR_SHAPE, "contextual_loss: the feature depth must be a multiple of 64");
  if (!(h > 0.f)) return fail(c, DVC_ERR_ARG, "contextual_loss: the bandwidth h must be > 0");
  if (c->corr_math == DVC_MATH_FP32) return fail(c, DVC_ERR_STATE, "contextual_loss: needs a tensor-core correlation mode");
  cudaStream_t s = (cudaStream_t)stream;
  CUDA_TRY(c, cudaSetDevice(c->device));
  void *mean, *xr, *yr, *V4, *y4, *m, *rsc, *den;
  DVC_TRY(get_raw(c, "ctx.mean", (size_t)B * C * 4, &mean, s));
  DVC_TRY(get_raw(c, "ctx.xrows", (size_t)B * NX * C * 4, &xr, s));
  DVC_TRY(get_raw(c, "ctx.yrows", (size_t)B * NY * C * 4, &yr, s));
  DVC_TRY(get_raw(c, "ctx.V4", (size_t)B * NY * 16, &V4, s));
  DVC_TRY(get_raw(c, "ctx.y4", (size_t)B * NX * 16, &y4, s));
  DVC_TRY(get_raw(c, "ctx.m", (size_t)B * NX * 4, &m, s));
  DVC_TRY(get_raw(c, "ctx.rsc", (size_t)B * NX * 4, &rsc, s));
  DVC_TRY(get_raw(c, "ctx.den", (size_t)B * NX * 4, &den, s));
  // both X and Y are centred by Y's channel means (ContextualLoss.py:99-104), then every position is scaled to unit norm
  if (feature_centering) {
    launch_chan_mean(dev_Y, (float*)mean, B, C, NY, s);
    DVC_TRY(check_launch(c, "chan_mean"));
  }
  const float eps = 2.220446049250313e-16f;
  launch_center_norm_rows(dev_X, feature_centering ? (const float*)mean : nullptr, (float*)xr, B, C, NX, eps, s);
  launch_center_norm_rows(dev_Y, feature_centering ? (const float*)mean : nullptr, (float*)yr, B, C, NY, eps, s);
  DVC_TRY(check_launch(c, "center_norm_rows"));
  launch_pack_v4(nullptr, (float*)V4, (size_t)B * NY, s);  // only the 4th lane (= 1) of the "colour" rows matters here
  CorrParams p{};
  p.theta = (float*)xr, p.phi = (float*)yr, p.V = (float*)V4, p.B = B, p.Bphi = B, p.NA = NX, p.NB = NY, p.C = C;
  p.y = (float*)y4, p.sim = (float*)m, p.argmax = nullptr;
  p.temperature = 1e-10f;  // pass 1: m_i = max_j f_ij
  DVC_TRY(run_corr(c, p, s));
  launch_ctx_row_scale((const float*)m, (float*)rsc, (size_t)B * NX, h, s);
  DVC_TRY(check_launch(c, "ctx_row_scale"));
  p.temperature = 1.0f, p.row_scale = (const float*)rsc, p.denom = (float*)den;  // pass 2: sum_j exp((f_ij - m_i) / T_i)
  DVC_TRY(run_corr(c, p, s));
  launch_ctx_loss((const float*)den, dev_loss, B, NX, s);
  return check_launch(c, "ctx_loss");
}

// ---- Fast Global Smoother ("WLS filter", test.py:105-112) ---------------------------------------------------------
// weights_LUT[d] = -exp(-d / sigma_color), d = |difference of neighbouring guide pixels|: evaluated in double and rounded
// once to the fp32 work type (the oracle does the same, so the two agree bit for bit).  Uploaded once per call.
static int fgs_lut(dvc_ctx* c, const std::string& name, float sigma_color, float** out, cudaStream_t s) {
  void* lut;
  DVC_TRY(get_raw(c, name, 256 * 4, &lut, s));
  float h_lut[256];
  for (int d = 0; d < 256; ++d) h_lut[d] = (float)(-exp(-(double)d / (double)sigma_color));
  CUDA_TRY(c, cudaMemcpyAsync(lut, h_lut, sizeof(h_lut), cudaMemcpyHostToDevice, s));
  CUDA_TRY(c, cudaStreamSynchronize(s));  // h_lut lives on this stack frame
  *out = (float*)lut;
  return DVC_OK;
}

// F frames of P planes x [F][P][H][W] filtered in place, frame f guided by guide [f] ([F][H][W]): one launch per step
static int fgs_run(dvc_ctx* c, const std::string& tag, const unsigned char* guide, float* x, int F, int P, int H, int W, float lambda,
                   const float* lut, float lambda_attenuation, int num_iter, cudaStream_t s) {
  const size_t hw = (size_t)H * W;
  void *Ch, *Cv, *D;
  DVC_TRY(get_raw(c, tag + ".Ch", (size_t)F * hw * 4, &Ch, s));
  DVC_TRY(get_raw(c, tag + ".Cv", (size_t)F * hw * 4, &Cv, s));
  DVC_TRY(get_raw(c, tag + ".D", (size_t)F * P * hw * 4, &D, s));
  launch_fgs_weights(guide, lut, (float*)Ch, (float*)Cv, F, H, W, s);
  DVC_TRY(check_launch(c, "fgs_weights"));
  float lam = lambda;
  for (int n = 0; n < num_iter; ++n) {
    launch_fgs_horizontal(x, (const float*)Ch, (float*)D, F * P, P, H, W, lam, s);
    launch_fgs_vertical(x, (const float*)Cv, (float*)D, F * P, P, H, W, lam, s);
    lam *= lambda_attenuation;
  }
  return check_launch(c, "fgs");
}

extern "C" int dvc_fgs_filter(dvc_ctx* c, const unsigned char* dev_guide, const float* dev_src, int planes, int H, int W, float lambda,
                              float sigma_color, float lambda_attenuation, int num_iter, float* dev_dst, void* stream) {
  if (!c || !dev_guide || !dev_src || !dev_dst || planes < 1 || H < 2 || W < 2) return c ? fail(c, DVC_ERR_ARG, "fgs_filter: bad argument") : DVC_ERR_ARG;
  if (!(lambda >= 0.f) || !(sigma_color > 0.f) || num_iter < 1 || !(lambda_attenuation > 0.f)) return fail(c, DVC_ERR_ARG, "fgs_filter: bad parameter");
  cudaStream_t s = (cudaStream_t)stream;
  CUDA_TRY(c, cudaSetDevice(c->device));
  float* lut;
  DVC_TRY(fgs_lut(c, "fgs.lut", sigma_color, &lut, s));
  if (dev_dst != dev_src) CUDA_TRY(c, cudaMemcpyAsync(dev_dst, dev_src, (size_t)planes * H * W * 4, cudaMemcpyDeviceToDevice, s));
  return fgs_run(c, "fgs", dev_guide, dev_dst, 1, planes, H, W, lambda, lut, lambda_attenuation, num_iter, s);
}

extern "C" int dvc_l_to_guide8(dvc_ctx* c, const float* dev_l, int H, int W, unsigned char* dev_guide, void* stream) {
  if (!c || !dev_l || !dev_guide || H < 1 || W < 1) return c ? fail(c, DVC_ERR_ARG, "l_to_guide8: bad argument") : DVC_ERR_ARG;
  CUDA_TRY(c, cudaSetDevice(c->device));
  launch_l_to_guide8(dev_l, dev_guide, (size_t)H * W, (cudaStream_t)stream);
  return check_launch(c, "l_to_guide8");
}

// ---- CenterPad's anti-aliased resize + crop / pad (util_distortion.py:217-258) ---------------------------------------
static void gaussian_taps(double sigma, std::vector<double>* w, int* radius) {  // scipy.ndimage._gaussian_kernel1d, truncate = 4
  const int r = (int)(4.0 * sigma + 0.5);
  w->assign(2 * r + 1, 0.0);
  const double s2 = sigma * sigma;
  double sum = 0.0;
  for (int x = -r; x <= r; ++x) (*w)[x + r] = exp(-0.5 / s2 * (double)(x * x)), sum += (*w)[x + r];
  for (double& v : *w) v /= sum;
  *radius = r;
}

// skimage.transform.resize's anti-aliasing Gaussians for an Hs x Ws -> Hr x Wr resize on the device: wy (2 ry + 1 taps),
// wx (2 rx + 1) and, at index 8191, a lone tap of weight 1 that converts uint8 -> float64 when the y axis needs no filter.
// Uploaded once per call (the host vectors live on this stack frame: the stream is synchronised).
struct ResizeTaps {
  const double *wy = nullptr, *wx = nullptr;
  int ry = 0, rx = 0;
};
static int resize_taps(dvc_ctx* c, const std::string& name, int Hs, int Ws, int Hr, int Wr, ResizeTaps* tp, cudaStream_t s) {
  void* taps;
  DVC_TRY(get_raw(c, name, 8192 * 8, &taps, s));
  // skimage.transform.resize: sigma = max(0, (in / out - 1) / 2) per axis, applied axis 0 first (scipy.ndimage.gaussian_filter)
  const double sy = fmax(0.0, ((double)Hs / Hr - 1.0) / 2.0), sx = fmax(0.0, ((double)Ws / Wr - 1.0) / 2.0);
  std::vector<double> wy, wx;
  int ry = 0, rx = 0;
  if (sy > 1e-15) gaussian_taps(sy, &wy, &ry);
  if (sx > 1e-15) gaussian_taps(sx, &wx, &rx);
  if (wy.size() + wx.size() > 8192) return fail(c, DVC_ERR_SHAPE, "resize_antialias_crop: down-scaling factor too large");
  const double one = 1.0;
  if (!wy.empty()) CUDA_TRY(c, cudaMemcpyAsync(taps, wy.data(), wy.size() * 8, cudaMemcpyHostToDevice, s));
  if (!wx.empty()) CUDA_TRY(c, cudaMemcpyAsync((double*)taps + wy.size(), wx.data(), wx.size() * 8, cudaMemcpyHostToDevice, s));
  if (wy.empty()) CUDA_TRY(c, cudaMemcpyAsync((double*)taps + 8191, &one, 8, cudaMemcpyHostToDevice, s));
  CUDA_TRY(c, cudaStreamSynchronize(s));
  tp->wy = wy.empty() ? (double*)taps + 8191 : (double*)taps, tp->ry = ry;
  tp->wx = wx.empty() ? nullptr : (double*)taps + wy.size(), tp->rx = rx;
  return DVC_OK;
}

// F uint8 frames [F][Hs][Ws][3] -> the anti-aliased float64 frames [F][Hs][Ws][3] (the Gaussian along y, then along x)
static int antialias_f64(dvc_ctx* c, const std::string& tag, const unsigned char* src, int F, int Hs, int Ws, const ResizeTaps& tp,
                         double** out, cudaStream_t s) {
  const size_t n = (size_t)F * Hs * Ws * 3;
  void *f0, *f1;
  DVC_TRY(get_raw(c, tag + ".f0", n * 8, &f0, s));
  DVC_TRY(get_raw(c, tag + ".f1", n * 8, &f1, s));
  double* cur = (double*)f0;
  double* nxt = (double*)f1;
  launch_gauss_axis_u8(src, cur, tp.wy, tp.ry, (size_t)F, Hs, Ws * 3, s);
  if (tp.wx) {
    launch_gauss_axis_f64(cur, nxt, tp.wx, tp.rx, (size_t)F * Hs, Ws, 3, s);
    std::swap(cur, nxt);
  }
  *out = cur;
  return check_launch(c, "antialias");
}

static bool bad_geometry(int Hs, int Ws, int Hr, int Wr, int Ho, int Wo) { return Hs < 1 || Ws < 1 || Hr < 1 || Wr < 1 || Ho < 1 || Wo < 1; }

extern "C" int dvc_resize_antialias_crop_rgb8(dvc_ctx* c, const unsigned char* dev_src, int Hs, int Ws, int Hr, int Wr, int oy, int ox,
                                              unsigned char* dev_dst, int Ho, int Wo, void* stream) {
  if (!c || !dev_src || !dev_dst || bad_geometry(Hs, Ws, Hr, Wr, Ho, Wo))
    return c ? fail(c, DVC_ERR_ARG, "resize_antialias_crop: bad argument") : DVC_ERR_ARG;
  cudaStream_t s = (cudaStream_t)stream;
  CUDA_TRY(c, cudaSetDevice(c->device));
  ResizeTaps tp;
  DVC_TRY(resize_taps(c, "rs.taps", Hs, Ws, Hr, Wr, &tp, s));
  double* cur;
  DVC_TRY(antialias_f64(c, "rs", dev_src, 1, Hs, Ws, tp, &cur, s));
  launch_zoom_crop(cur, Hs, Ws, Hr, Wr, oy, ox, dev_dst, Ho, Wo, s);
  return check_launch(c, "resize_antialias_crop");
}

// ---- whole frames in, whole frames out ---------------------------------------------------------------------------------
static int ingest_enqueue(dvc_ctx* c, const std::string& tag, const unsigned char* src, int F, int Hs, int Ws, int Hr, int Wr, int oy,
                          int ox, int Ho, int Wo, const ResizeTaps& tp, float* l, float* l_half, cudaStream_t s) {
  double* cur;
  DVC_TRY(antialias_f64(c, tag, src, F, Hs, Ws, tp, &cur, s));
  launch_ingest_l(cur, F, Hs, Ws, Hr, Wr, oy, ox, l, Ho, Wo, s);
  launch_resize_half(l, l_half, F, Ho, Wo, s);  // test.py:71
  return check_launch(c, "ingest");
}

static int postprocess_enqueue(dvc_ctx* c, const std::string& tag, const float* l, const float* ab_half, int F, int Ho, int Wo, int wls,
                               float lambda, const float* lut, unsigned char* rgb, cudaStream_t s) {
  const size_t hw = (size_t)Ho * Wo;
  void *up, *guide;
  DVC_TRY(get_raw(c, tag + ".up", (size_t)F * 2 * hw * 4, &up, s));
  launch_upsample2(ab_half, (float*)up, F * 2, Ho / 2, Wo / 2, 1.25f, s);  // test.py:100-102
  if (wls) {                                                              // test.py:105-112
    DVC_TRY(get_raw(c, tag + ".guide", (size_t)F * hw, &guide, s));
    launch_l_to_guide8(l, (unsigned char*)guide, (size_t)F * hw, s);
    DVC_TRY(fgs_run(c, tag, (const unsigned char*)guide, (float*)up, F, 2, Ho, Wo, lambda, lut, 0.25f, 3, s));
  }
  double inv[9];
  rgb_from_xyz(inv);
  launch_lab_to_rgb8(l, (const float*)up, rgb, F, Ho, Wo, inv, s);  // test.py:116-119
  return check_launch(c, "postprocess");
}

static bool bad_out_size(int Ho, int Wo) { return Ho < 2 || Wo < 2 || (Ho & 1) || (Wo & 1); }
static int check_wls(dvc_ctx* c, float lambda, float sigma_color) {
  if (!(lambda >= 0.f) || !(sigma_color > 0.f)) return fail(c, DVC_ERR_ARG, "WLS filter: lambda must be >= 0 and sigma_color > 0");
  return DVC_OK;
}

extern "C" int dvc_ingest_rgb8(dvc_ctx* c, const unsigned char* dev_src, int F, int Hs, int Ws, int Hr, int Wr, int oy, int ox, int Ho,
                               int Wo, float* dev_l, float* dev_l_half, void* stream) {
  if (!c || !dev_src || !dev_l || !dev_l_half || F < 1 || bad_geometry(Hs, Ws, Hr, Wr, Ho, Wo))
    return c ? fail(c, DVC_ERR_ARG, "ingest_rgb8: bad argument") : DVC_ERR_ARG;
  if (bad_out_size(Ho, Wo)) return fail(c, DVC_ERR_SHAPE, "ingest_rgb8: Ho and Wo must be even");
  cudaStream_t s = (cudaStream_t)stream;
  CUDA_TRY(c, cudaSetDevice(c->device));
  ResizeTaps tp;
  DVC_TRY(resize_taps(c, "ing.taps", Hs, Ws, Hr, Wr, &tp, s));
  return ingest_enqueue(c, "ing", dev_src, F, Hs, Ws, Hr, Wr, oy, ox, Ho, Wo, tp, dev_l, dev_l_half, s);
}

extern "C" int dvc_postprocess_rgb8(dvc_ctx* c, const float* dev_l, const float* dev_ab_half, int F, int Ho, int Wo, int wls, float lambda,
                                    float sigma_color, unsigned char* dev_rgb, void* stream) {
  if (!c || !dev_l || !dev_ab_half || !dev_rgb || F < 1) return c ? fail(c, DVC_ERR_ARG, "postprocess_rgb8: bad argument") : DVC_ERR_ARG;
  if (bad_out_size(Ho, Wo)) return fail(c, DVC_ERR_SHAPE, "postprocess_rgb8: Ho and Wo must be even");
  if (wls) DVC_TRY(check_wls(c, lambda, sigma_color));
  cudaStream_t s = (cudaStream_t)stream;
  CUDA_TRY(c, cudaSetDevice(c->device));
  float* lut = nullptr;
  if (wls) DVC_TRY(fgs_lut(c, "post.lut", sigma_color, &lut, s));
  return postprocess_enqueue(c, "post", dev_l, dev_ab_half, F, Ho, Wo, wls, lambda, lut, dev_rgb, s);
}

// The clip driver with uint8 frames on both ends.  Rings (device memory depends on the frame sizes and G only):
//   source frame  1 slot  (H2D and ingest are ordered on the upload stream)
//   full-size L   2G slots  } batch b of G frames uses slot half b & 1; written by ingest / ColorVidNet, read by the
//   half-size ab  2G slots  } batch's post-processing, reused by batch b + 2 after evP[b & 1]
//   RGB           G slots   (post-processing and the download are ordered on the post stream)
extern "C" int dvc_colorize_video_rgb8(dvc_ctx* c, const unsigned char* host_src, int K, int Hs, int Ws, int Hr, int Wr, int oy, int ox,
                                       int Ho, int Wo, float temperature, int wls, float lambda, float sigma_color, int continue_clip,
                                       unsigned char* host_dst, void* stream) {
  if (!c || !host_src || !host_dst || K < 1 || bad_geometry(Hs, Ws, Hr, Wr, Ho, Wo))
    return c ? fail(c, DVC_ERR_ARG, "colorize_video_rgb8: bad argument") : DVC_ERR_ARG;
  if (bad_out_size(Ho, Wo)) return fail(c, DVC_ERR_SHAPE, "colorize_video_rgb8: Ho and Wo must be even");
  if (wls) DVC_TRY(check_wls(c, lambda, sigma_color));
  const int H = Ho / 2, W = Wo / 2;
  DVC_TRY(check_frame_args(c, H, W, temperature));
  if (continue_clip && (c->vid_ex_version != c->ex_version || c->vid_Ho != Ho || c->vid_Wo != Wo))
    return fail(c, DVC_ERR_STATE, "colorize_video_rgb8: nothing to continue (no earlier call against this exemplar at this size)");
  cudaStream_t s = (cudaStream_t)stream;
  CUDA_TRY(c, cudaSetDevice(c->device));
  DVC_TRY(clip_streams(c));
  const int G = c->video_batch;
  const size_t hw = (size_t)H * W, HW = (size_t)Ho * Wo, src_bytes = (size_t)Hs * Ws * 3;
  void *dlast, *dsrc, *dLf, *dab, *drgb;
  DVC_TRY(get_raw(c, "vid.last", 3 * hw * 4, &dlast, s));
  DVC_TRY(get_raw(c, "vid.src", src_bytes, &dsrc, s));
  DVC_TRY(get_raw(c, "vid.Lfull", (size_t)2 * G * HW * 4, &dLf, s));
  DVC_TRY(get_raw(c, "vid.ab", (size_t)2 * G * 2 * hw * 4, &dab, s));
  DVC_TRY(get_raw(c, "vid.rgb", (size_t)G * HW * 3, &drgb, s));
  {  // post-processing work buffers at their full batch size now: growing one inside the frame loop would cudaFree it
    void* p;
    DVC_TRY(get_raw(c, "vid.up", (size_t)G * 2 * HW * 4, &p, s));
    DVC_TRY(get_raw(c, "vid.guide", (size_t)G * HW, &p, s));
    DVC_TRY(get_raw(c, "vid.Ch", (size_t)G * HW * 4, &p, s));
    DVC_TRY(get_raw(c, "vid.Cv", (size_t)G * HW * 4, &p, s));
    DVC_TRY(get_raw(c, "vid.D", (size_t)G * 2 * HW * 4, &p, s));
  }
  ResizeTaps tp;
  DVC_TRY(resize_taps(c, "vid.taps", Hs, Ws, Hr, Wr, &tp, s));
  float* lut = nullptr;
  if (wls) DVC_TRY(fgs_lut(c, "vid.lut", sigma_color, &lut, s));
  c->vid_ex_version = -1;  // valid again only once this call has succeeded
  if (!continue_clip) CUDA_TRY(c, cudaMemsetAsync(dlast, 0, 3 * hw * 4, s));  // test.py:80
  float* Lfull = (float*)dLf;
  float* ab = (float*)dab;
  ClipStages st;
  st.ingest = [&](int t, float* Lt, cudaStream_t su) -> int {
    if (t >= 2 * G) CUDA_TRY(c, cudaStreamWaitEvent(su, c->evP[(t / G) & 1], 0));  // batch t / G - 2 is post-processed
    CUDA_TRY(c, cudaMemcpyAsync(dsrc, host_src + (size_t)t * src_bytes, src_bytes, cudaMemcpyDefault, su));
    return ingest_enqueue(c, "vid", (const unsigned char*)dsrc, 1, Hs, Ws, Hr, Wr, oy, ox, Ho, Wo, tp, Lfull + (size_t)(t % (2 * G)) * HW,
                          Lt, su);
  };
  st.ab_slot = [&](int t, cudaStream_t sc, float** abt) -> int {
    if (t >= 2 * G) CUDA_TRY(c, cudaStreamWaitEvent(sc, c->evP[(t / G) & 1], 0));
    *abt = ab + (size_t)(t % (2 * G)) * 2 * hw;
    return DVC_OK;
  };
  st.egress = [&](int t, const float*, cudaEvent_t done) -> int {
    if (t % G != G - 1 && t != K - 1) return DVC_OK;  // post-processing runs once per batch
    const int n = t % G + 1, t0 = t + 1 - n, slot = t0 % (2 * G);
    CUDA_TRY(c, cudaStreamWaitEvent(c->sP, done, 0));
    DVC_TRY(postprocess_enqueue(c, "vid", Lfull + (size_t)slot * HW, ab + (size_t)slot * 2 * hw, n, Ho, Wo, wls, lambda, lut,
                                (unsigned char*)drgb, c->sP));
    CUDA_TRY(c, cudaMemcpyAsync(host_dst + (size_t)t0 * HW * 3, drgb, (size_t)n * HW * 3, cudaMemcpyDefault, c->sP));
    CUDA_TRY(c, cudaEventRecord(c->evP[(t / G) & 1], c->sP));
    return DVC_OK;
  };
  DVC_TRY(run_clip(c, K, H, W, temperature, (float*)dlast, st, s));
  c->vid_ex_version = c->ex_version, c->vid_Ho = Ho, c->vid_Wo = Wo;
  return DVC_OK;
}

// ---- exemplar operands for the NCCL broadcast -----------------------------------------------------
extern "C" int64_t dvc_exemplar_pack_size(const dvc_ctx*, int H, int W) {
  const int64_t N = (int64_t)(H / 4) * (W / 4);
  return N * 256 + N * 4;
}

extern "C" int dvc_exemplar_export(dvc_ctx* c, float* buf, int64_t n, void* stream) {
  if (!c || !buf) return c ? fail(c, DVC_ERR_ARG, "exemplar_export: bad argument") : DVC_ERR_ARG;
  if (!c->ex_valid) return fail(c, DVC_ERR_STATE, "exemplar_export: no exemplar set");
  const int64_t N = c->ex_N;
  if (n != N * 260) return fail(c, DVC_ERR_SHAPE, "exemplar_export: buffer size mismatch");
  cudaStream_t s = (cudaStream_t)stream;
  CUDA_TRY(c, cudaMemcpyAsync(buf, c->ex_phi, (size_t)N * 256 * 4, cudaMemcpyDeviceToDevice, s));
  CUDA_TRY(c, cudaMemcpyAsync(buf + N * 256, c->ex_V, (size_t)N * 16, cudaMemcpyDeviceToDevice, s));
  return DVC_OK;
}

extern "C" int dvc_exemplar_import(dvc_ctx* c, const float* buf, int64_t n, int H, int W, void* stream) {
  if (!c || !buf) return c ? fail(c, DVC_ERR_ARG, "exemplar_import: bad argument") : DVC_ERR_ARG;
  if (!legal_shape(H, W)) return fail(c, DVC_ERR_SHAPE, "exemplar_import: illegal frame shape");
  const int64_t N = (int64_t)(H / 4) * (W / 4);
  if (n != N * 260) return fail(c, DVC_ERR_SHAPE, "exemplar_import: buffer size mismatch");
  cudaStream_t s = (cudaStream_t)stream;
  CUDA_TRY(c, cudaSetDevice(c->device));
  if (c->ex_N != N) {
    if (c->ex_phi) cudaFree(c->ex_phi);
    if (c->ex_V) cudaFree(c->ex_V);
    c->ex_phi = c->ex_V = nullptr;
    CUDA_TRY(c, cudaMalloc((void**)&c->ex_phi, (size_t)N * 256 * 4));
    CUDA_TRY(c, cudaMalloc((void**)&c->ex_V, (size_t)N * 16));
    c->ex_N = (int)N;
  }
  CUDA_TRY(c, cudaMemcpyAsync(c->ex_phi, buf, (size_t)N * 256 * 4, cudaMemcpyDeviceToDevice, s));
  CUDA_TRY(c, cudaMemcpyAsync(c->ex_V, buf + N * 256, (size_t)N * 16, cudaMemcpyDeviceToDevice, s));
  // whatever produced the pack, the 4th lane of every V row must be 1 (corr_tc.cu's softmax epilogue)
  launch_pack_v4(nullptr, c->ex_V, (size_t)N, s);
  DVC_TRY(check_launch(c, "pack_v4"));
  c->ex_H = H, c->ex_W = W, c->ex_valid = true, c->ex_version++;
  if (corr_ws_reserve(&c->corr_ws, 1, 1, (int)N, (int)N) != 0) return fail(c, DVC_ERR_CUDA, "exemplar_import: correlation workspace allocation failed");
  return DVC_OK;
}
