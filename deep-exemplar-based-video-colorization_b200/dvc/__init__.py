"""ctypes binding of libdvc.so (include/dvc.h) -- the only way Python reaches the CUDA kernels.

PyTorch is used for device memory, streams and torch.distributed; every FLOP of the hot path runs
in hand-written sm_100a kernels inside libdvc.so.  There is no CPU fallback and no torch fallback:
if the library or a CUDA device is missing, every entry point raises.
"""
import ctypes
import os
import threading

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(os.path.dirname(_HERE), "lib", "libdvc.so")

NET_VGG, NET_WARP, NET_COLOR = 0, 1, 2
MATH_FP32, MATH_TF32X3, MATH_BF16X3, MATH_FP16X3 = 0, 1, 2, 3

EXPORTED = [
    "dvc_create", "dvc_destroy", "dvc_last_error", "dvc_version", "dvc_set_math", "dvc_set_weight",
    "dvc_vgg19_forward", "dvc_warpnet_forward", "dvc_colorvidnet_forward", "dvc_corr_softmax_warp",
    "dvc_set_exemplar", "dvc_colorize_frames", "dvc_colorize_clip", "dvc_exemplar_pack_size",
    "dvc_exemplar_export", "dvc_exemplar_import", "dvc_launch_count", "dvc_profile_corr", "dvc_corr_mean_ms",
    "dvc_debug_set_flag", "dvc_debug_get_buffer", "dvc_debug_conv2d", "dvc_profile_conv", "dvc_conv_profile",
    "dvc_resize_half", "dvc_upsample2_scaled", "dvc_lab_to_rgb8", "dvc_rgb8_to_lab",
    "dvc_fgs_filter", "dvc_l_to_guide8", "dvc_resize_antialias_crop_rgb8", "dvc_contextual_loss_forward",
    "dvc_peer_buffer_create", "dvc_peer_buffer_open", "dvc_peer_buffer_close", "dvc_peer_buffer_destroy",
    "dvc_corr_set_peer_outputs", "dvc_ingest_rgb8", "dvc_postprocess_rgb8", "dvc_colorize_video_rgb8",
]

_lib = None
_lib_lock = threading.Lock()


class DvcError(RuntimeError):
    pass


def load_library():
    """dlopen libdvc.so and declare the prototypes of include/dvc.h.  Fails loudly if it is not built."""
    global _lib
    with _lib_lock:
        if _lib is not None:
            return _lib
        if not os.path.isfile(LIB_PATH):
            raise DvcError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(there is no fallback implementation)")
        lib = ctypes.CDLL(LIB_PATH)
        c_void, c_int, c_float, c_i64 = ctypes.c_void_p, ctypes.c_int, ctypes.c_float, ctypes.c_int64
        P = ctypes.POINTER
        lib.dvc_create.argtypes = [P(c_void), c_int]
        lib.dvc_destroy.argtypes = [c_void]
        lib.dvc_last_error.argtypes = [c_void]
        lib.dvc_last_error.restype = ctypes.c_char_p
        lib.dvc_version.restype = ctypes.c_char_p
        lib.dvc_set_math.argtypes = [c_void, c_int, c_int]
        lib.dvc_set_weight.argtypes = [c_void, c_int, ctypes.c_char_p, c_void, P(c_i64), c_int]
        lib.dvc_vgg19_forward.argtypes = [c_void, c_void, c_int, c_int, c_int, c_int, P(ctypes.c_char_p), P(c_void),
                                          c_int, c_void]
        lib.dvc_warpnet_forward.argtypes = [c_void, c_void, P(c_void), P(c_void), c_int, c_int, c_int, c_float, c_float,
                                            c_int, c_void, c_void, c_void]
        lib.dvc_colorvidnet_forward.argtypes = [c_void, c_void, c_int, c_int, c_int, c_void, c_void]
        lib.dvc_corr_softmax_warp.argtypes = [c_void, c_void, c_void, c_void, c_int, c_int, c_int, c_int, c_int, c_float,
                                              c_void, c_void, c_void, c_void]
        lib.dvc_set_exemplar.argtypes = [c_void, c_void, c_int, c_int, c_void]
        lib.dvc_colorize_frames.argtypes = [c_void, c_void, c_void, c_int, c_int, c_int, c_float, c_void, c_void, c_void,
                                            c_void]
        lib.dvc_colorize_clip.argtypes = [c_void, c_void, c_int, c_int, c_int, c_float, c_void, c_void, c_void]
        lib.dvc_exemplar_pack_size.argtypes = [c_void, c_int, c_int]
        lib.dvc_exemplar_pack_size.restype = c_i64
        lib.dvc_exemplar_export.argtypes = [c_void, c_void, c_i64, c_void]
        lib.dvc_exemplar_import.argtypes = [c_void, c_void, c_i64, c_int, c_int, c_void]
        lib.dvc_launch_count.argtypes = [c_void, c_int]
        lib.dvc_launch_count.restype = c_i64
        lib.dvc_profile_corr.argtypes = [c_void, c_int]
        lib.dvc_corr_mean_ms.argtypes = [c_void, c_int]
        lib.dvc_corr_mean_ms.restype = ctypes.c_double
        lib.dvc_resize_half.argtypes = [c_void, c_void, c_int, c_int, c_int, c_void, c_void]
        lib.dvc_upsample2_scaled.argtypes = [c_void, c_void, c_int, c_int, c_int, c_float, c_void, c_void]
        lib.dvc_lab_to_rgb8.argtypes = [c_void, c_void, c_void, c_int, c_int, c_int, c_void, c_void]
        lib.dvc_rgb8_to_lab.argtypes = [c_void, c_void, c_int, c_int, c_int, c_void, c_void]
        lib.dvc_fgs_filter.argtypes = [c_void, c_void, c_void, c_int, c_int, c_int, c_float, c_float, c_float, c_int, c_void, c_void]
        lib.dvc_l_to_guide8.argtypes = [c_void, c_void, c_int, c_int, c_void, c_void]
        lib.dvc_resize_antialias_crop_rgb8.argtypes = [c_void, c_void, c_int, c_int, c_int, c_int, c_int, c_int, c_void, c_int, c_int,
                                                       c_void]
        lib.dvc_ingest_rgb8.argtypes = [c_void, c_void] + [c_int] * 9 + [c_void, c_void, c_void]
        lib.dvc_postprocess_rgb8.argtypes = [c_void, c_void, c_void, c_int, c_int, c_int, c_int, c_float, c_float, c_void, c_void]
        lib.dvc_colorize_video_rgb8.argtypes = ([c_void, c_void] + [c_int] * 9 + [c_float, c_int, c_float, c_float, c_int]
                                                + [c_void, c_void])
        lib.dvc_contextual_loss_forward.argtypes = [c_void, c_void, c_void, c_int, c_int, c_int, c_int, c_float, c_int, c_void, c_void]
        lib.dvc_peer_buffer_create.argtypes = [c_void, c_i64, P(c_void), ctypes.c_char_p]
        lib.dvc_peer_buffer_open.argtypes = [c_void, ctypes.c_char_p, P(c_void)]
        lib.dvc_peer_buffer_close.argtypes = [c_void, c_void]
        lib.dvc_peer_buffer_destroy.argtypes = [c_void, c_void]
        lib.dvc_corr_set_peer_outputs.argtypes = [c_void, c_int, P(c_void), P(c_void), c_i64]
        lib.dvc_profile_conv.argtypes = [c_void, c_int]
        lib.dvc_conv_profile.argtypes = [c_void, c_int, c_int, P(ctypes.c_double), P(ctypes.c_double)]
        lib.dvc_debug_set_flag.argtypes = [c_void, ctypes.c_char_p, c_int]
        lib.dvc_debug_get_buffer.argtypes = [c_void, ctypes.c_char_p, P(c_void), P(c_i64), P(c_int)]
        lib.dvc_debug_conv2d.argtypes = [c_void, c_int, ctypes.c_char_p, c_void, c_int, c_int, c_int, c_int, c_int, c_int, c_float,
                                         c_int, c_int, c_int, c_float, c_int, c_void, c_void, c_void, c_void]
        _lib = lib
        return lib


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)


def _stream(device):
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _dev_f32(t, what):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise DvcError(f"{what}: expected a CUDA tensor (libdvc has no CPU path)")
    if t.dtype != torch.float32:
        raise DvcError(f"{what}: expected float32, got {t.dtype}")
    return t.contiguous()


class Context:
    """One dvc_ctx per CUDA device; owns the weights of all three networks and all workspaces."""

    def __init__(self, device=0):
        self.lib = load_library()
        if not torch.cuda.is_available():
            raise DvcError("no CUDA device visible: libdvc has no CPU fallback")
        self.device = torch.device("cuda", device if isinstance(device, int) else torch.device(device).index or 0)
        h = ctypes.c_void_p(0)
        rc = self.lib.dvc_create(ctypes.byref(h), self.device.index)
        if rc != 0:
            raise DvcError(f"dvc_create failed ({rc}): {self.lib.dvc_last_error(None).decode()}")
        self.h = h
        self._weight_sig = {}

    def close(self):
        if getattr(self, "h", None):
            self.lib.dvc_destroy(self.h)
            self.h = None

    def _check(self, rc, what):
        if rc != 0:
            raise DvcError(f"{what} failed ({rc}): {self.lib.dvc_last_error(self.h).decode()}")

    # ---- configuration / weights -------------------------------------------------------------
    def set_math(self, conv=MATH_TF32X3, corr=MATH_FP16X3):
        self._check(self.lib.dvc_set_math(self.h, conv, corr), "dvc_set_math")

    def set_weights(self, net, state_dict):
        """Replaces load_state_dict (test.py:150,158-159) for `net` in {NET_VGG, NET_WARP, NET_COLOR}."""
        self._weight_sig.pop(net, None)  # a drop-in module that synced earlier must re-upload on its next forward
        for key, t in state_dict.items():
            t = t.detach().to(torch.float32).contiguous()
            shape = (ctypes.c_int64 * t.dim())(*t.shape)
            self._check(self.lib.dvc_set_weight(self.h, net, key.encode(), _ptr(t), shape, t.dim()),
                        f"dvc_set_weight({key})")

    def sync_module_weights(self, net, module):
        """Push a drop-in module's parameters when they changed (load_state_dict / .cuda() / in-place edit)."""
        sd = module.state_dict()
        sig = tuple((k, v.data_ptr(), v._version, tuple(v.shape)) for k, v in sd.items())
        if self._weight_sig.get(net) != sig:
            self.set_weights(net, sd)
            self._weight_sig[net] = sig

    # ---- module-level drop-ins -----------------------------------------------------------------
    def vgg19_forward(self, x, out_keys, preprocess=True):
        x = _dev_f32(x, "VGG19 input")
        if x.dim() != 4 or x.shape[1] != 3:
            raise DvcError("VGG19 input must be [B,3,H,W]")
        B, _, H, W = x.shape
        dims = {}
        h, w = H, W
        chans = [64, 128, 256, 512, 512]
        nconv = [2, 2, 4, 4, 4]
        for blk in range(5):
            for i in range(nconv[blk]):
                dims[f"r{blk + 1}{i + 1}"] = (chans[blk], h, w)
            h, w = h // 2, w // 2
            dims[f"p{blk + 1}"] = (chans[blk], h, w)
        outs = []
        for k in out_keys:
            if k not in dims:
                raise DvcError(f"unknown VGG key {k!r}")
            c, hh, ww = dims[k]
            outs.append(torch.empty(B, c, hh, ww, device=x.device, dtype=torch.float32))
        keys = (ctypes.c_char_p * len(out_keys))(*[k.encode() for k in out_keys])
        ptrs = (ctypes.c_void_p * len(outs))(*[o.data_ptr() for o in outs])
        rc = self.lib.dvc_vgg19_forward(self.h, _ptr(x), B, H, W, 1 if preprocess else 0, keys, ptrs, len(outs),
                                        _stream(x.device))
        self._check(rc, "dvc_vgg19_forward")
        return outs

    def warpnet_forward(self, B_lab_map, A_feats, B_feats, temperature, wta_scale_weight=1.0, reuse_exemplar=False):
        B_lab_map = _dev_f32(B_lab_map, "B_lab_map")
        A = [_dev_f32(t, "A feature") for t in A_feats]
        Bf = [_dev_f32(t, "B feature") for t in B_feats]
        Bn, ch, H, W = B_lab_map.shape
        if ch != 3:
            raise DvcError("B_lab_map must have 3 channels")
        y = torch.empty(Bn, 3, H, W, device=B_lab_map.device, dtype=torch.float32)
        sim = torch.empty(Bn, 1, H, W, device=B_lab_map.device, dtype=torch.float32)
        pa = (ctypes.c_void_p * 4)(*[t.data_ptr() for t in A])
        pb = (ctypes.c_void_p * 4)(*[t.data_ptr() for t in Bf])
        rc = self.lib.dvc_warpnet_forward(self.h, _ptr(B_lab_map), pa, pb, Bn, H, W, float(temperature),
                                          float(wta_scale_weight), 1 if reuse_exemplar else 0, _ptr(y), _ptr(sim),
                                          _stream(B_lab_map.device))
        self._check(rc, "dvc_warpnet_forward")
        return y, sim

    def colorvidnet_forward(self, x):
        x = _dev_f32(x, "ColorVidNet input")
        if x.dim() != 4 or x.shape[1] != 7:
            raise DvcError("ColorVidNet input must be [B,7,H,W]")
        B, _, H, W = x.shape
        out = torch.empty(B, 2, H, W, device=x.device, dtype=torch.float32)
        self._check(self.lib.dvc_colorvidnet_forward(self.h, _ptr(x), B, H, W, _ptr(out), _stream(x.device)),
                    "dvc_colorvidnet_forward")
        return out

    def corr_softmax_warp(self, theta_hat, phi_hat, V, temperature, want_argmax=False):
        """theta_hat [B,C,NA], phi_hat [Bphi,C,NB], V [Bphi,NB,3] -> y [B,NA,3], sim [B,NA] (, argmax)."""
        theta_hat, phi_hat, V = _dev_f32(theta_hat, "theta_hat"), _dev_f32(phi_hat, "phi_hat"), _dev_f32(V, "V")
        B, C, NA = theta_hat.shape
        Bphi, _, NB = phi_hat.shape
        y = torch.empty(B, NA, 3, device=theta_hat.device, dtype=torch.float32)
        sim = torch.empty(B, NA, device=theta_hat.device, dtype=torch.float32)
        am = torch.empty(B, NA, device=theta_hat.device, dtype=torch.int32) if want_argmax else None
        rc = self.lib.dvc_corr_softmax_warp(self.h, _ptr(theta_hat), _ptr(phi_hat), _ptr(V), B, Bphi, NA, NB, C,
                                            float(temperature), _ptr(y), _ptr(sim), _ptr(am), _stream(theta_hat.device))
        self._check(rc, "dvc_corr_softmax_warp")
        return (y, sim, am) if want_argmax else (y, sim)

    # ---- fused per-frame / per-clip path ---------------------------------------------------------
    def set_exemplar(self, IB_lab):
        t = IB_lab.detach().to(torch.float32).contiguous()
        if t.dim() != 4 or t.shape[0] != 1 or t.shape[1] != 3:
            raise DvcError("exemplar must be [1,3,H,W]")
        self._check(self.lib.dvc_set_exemplar(self.h, _ptr(t), t.shape[2], t.shape[3], _stream(self.device)),
                    "dvc_set_exemplar")
        if not t.is_cuda:
            torch.cuda.current_stream(self.device).synchronize()  # the host buffer must outlive the async copy

    def colorize_frames(self, IA_l, IA_last_lab, temperature=1e-10, want_warp=False):
        IA_l, IA_last_lab = _dev_f32(IA_l, "IA_l"), _dev_f32(IA_last_lab, "IA_last_lab")
        B, c1, H, W = IA_l.shape
        if c1 != 1 or tuple(IA_last_lab.shape) != (B, 3, H, W):
            raise DvcError("IA_l must be [B,1,H,W] and IA_last_lab [B,3,H,W]")
        ab = torch.empty(B, 2, H, W, device=IA_l.device, dtype=torch.float32)
        warp = torch.empty(B, 3, H, W, device=IA_l.device, dtype=torch.float32) if want_warp else None
        sim = torch.empty(B, 1, H, W, device=IA_l.device, dtype=torch.float32) if want_warp else None
        rc = self.lib.dvc_colorize_frames(self.h, _ptr(IA_l), _ptr(IA_last_lab), B, H, W, float(temperature), _ptr(ab),
                                          _ptr(warp), _ptr(sim), _stream(IA_l.device))
        self._check(rc, "dvc_colorize_frames")
        return (ab, warp, sim) if want_warp else ab

    def colorize_clip(self, L, temperature=1e-10, first_last_lab=None, out=None):
        """L [F,1,H,W] -> ab [F,2,H,W] with the recurrence of test.py:76-96 kept on the device.

        L may be a pinned CPU tensor (one host->device copy of L and one device->host copy of ab per frame inside
        the call) or a CUDA tensor (frames already resident in HBM); `out` lives where L lives."""
        if L.dtype != torch.float32 or L.dim() != 4 or L.shape[1] != 1:
            raise DvcError("colorize_clip takes a float32 [F,1,H,W] tensor")
        L = L.contiguous()
        F_, _, H, W = L.shape
        if out is None:
            out = torch.empty(F_, 2, H, W, dtype=torch.float32, device=L.device)
            if not L.is_cuda:
                out = out.pin_memory()
        if out.is_cuda != L.is_cuda or not out.is_contiguous() or tuple(out.shape) != (F_, 2, H, W):
            raise DvcError("colorize_clip: `out` must be a contiguous [F,2,H,W] tensor on the same side as L")
        fl = first_last_lab.contiguous() if first_last_lab is not None else None
        rc = self.lib.dvc_colorize_clip(self.h, _ptr(L), F_, H, W, float(temperature), _ptr(fl), _ptr(out),
                                        _stream(self.device))
        self._check(rc, "dvc_colorize_clip")
        return out

    # ---- pre / post-processing around the nets (test.py:58,71,100-102) ----------------------------------
    def resize_half(self, x):
        """F.interpolate(x, scale_factor=0.5, mode="bilinear") for a CUDA [B,C,H,W] tensor with even H, W."""
        x = _dev_f32(x, "resize_half input")
        B, C, H, W = x.shape
        out = torch.empty(B, C, H // 2, W // 2, device=x.device, dtype=torch.float32)
        self._check(self.lib.dvc_resize_half(self.h, _ptr(x), B * C, H, W, _ptr(out), _stream(x.device)), "dvc_resize_half")
        return out

    def upsample2_scaled(self, x, scale=1.25):
        """F.interpolate(x, scale_factor=2, mode="bilinear") * scale for a CUDA [B,C,h,w] tensor."""
        x = _dev_f32(x, "upsample2 input")
        B, C, h, w = x.shape
        out = torch.empty(B, C, 2 * h, 2 * w, device=x.device, dtype=torch.float32)
        self._check(self.lib.dvc_upsample2_scaled(self.h, _ptr(x), B * C, h, w, float(scale), _ptr(out), _stream(x.device)),
                    "dvc_upsample2_scaled")
        return out

    def lab_to_rgb8(self, l, ab):
        """batch_lab2rgb_transpose_mc (utils/util.py:140-151) for CUDA l [B,1,H,W] (centred) and ab [B,2,H,W]:
        uint8 [B,H,W,3] sRGB, computed in float64 like skimage.color.lab2rgb."""
        l, ab = _dev_f32(l, "lab_to_rgb8 l"), _dev_f32(ab, "lab_to_rgb8 ab")
        B, _, H, W = l.shape
        if tuple(ab.shape) != (B, 2, H, W) or l.shape[1] != 1:
            raise DvcError("lab_to_rgb8: expected l [B,1,H,W] and ab [B,2,H,W]")
        out = torch.empty(B, H, W, 3, device=l.device, dtype=torch.uint8)
        self._check(self.lib.dvc_lab_to_rgb8(self.h, _ptr(l), _ptr(ab), B, H, W, ctypes.c_void_p(out.data_ptr()), _stream(l.device)),
                    "dvc_lab_to_rgb8")
        return out

    def rgb8_to_lab(self, rgb):
        """RGB2Lab + ToTensor + Normalize of test.py:44-45 for a CUDA uint8 [B,H,W,3] tensor: float32 [B,3,H,W] with
        centred L, computed in float64 like skimage.color.rgb2lab."""
        if not (isinstance(rgb, torch.Tensor) and rgb.is_cuda and rgb.dtype == torch.uint8 and rgb.dim() == 4 and rgb.shape[3] == 3):
            raise DvcError("rgb8_to_lab: expected a CUDA uint8 tensor [B,H,W,3]")
        rgb = rgb.contiguous()
        B, H, W, _ = rgb.shape
        out = torch.empty(B, 3, H, W, device=rgb.device, dtype=torch.float32)
        self._check(self.lib.dvc_rgb8_to_lab(self.h, ctypes.c_void_p(rgb.data_ptr()), B, H, W, _ptr(out), _stream(rgb.device)),
                    "dvc_rgb8_to_lab")
        return out

    def contextual_loss_forward(self, X_features, Y_features, h=0.1, feature_centering=True):
        """ContextualLoss_forward.forward (models/ContextualLoss.py:82-126), value only: CUDA float32 [B,C,h,w] (or [B,C,N])
        feature maps -> loss [B]."""
        X, Y = _dev_f32(X_features, "contextual_loss X"), _dev_f32(Y_features, "contextual_loss Y")
        B, C = X.shape[0], X.shape[1]
        if Y.shape[0] != B or Y.shape[1] != C:
            raise DvcError("contextual_loss: X and Y must share batch size and feature depth")
        NX, NY = X[0, 0].numel(), Y[0, 0].numel()
        out = torch.empty(B, device=X.device, dtype=torch.float32)
        self._check(self.lib.dvc_contextual_loss_forward(self.h, _ptr(X), _ptr(Y), B, C, NX, NY, float(h), 1 if feature_centering else 0,
                                                         _ptr(out), _stream(X.device)), "dvc_contextual_loss_forward")
        return out

    def fgs_filter(self, guide, src, lam=500.0, sigma_color=4.0, lambda_attenuation=0.25, num_iter=3):
        """cv2.ximgproc.createFastGlobalSmootherFilter(guide, lam, sigma_color).filter(plane) for every plane of the
        CUDA float32 tensor src [P,H,W] with the CUDA uint8 guide [H,W] (test.py:105-112; defaults of test.py:32-33)."""
        src = _dev_f32(src, "fgs_filter src")
        if not (isinstance(guide, torch.Tensor) and guide.is_cuda and guide.dtype == torch.uint8 and guide.dim() == 2):
            raise DvcError("fgs_filter: the guide must be a CUDA uint8 [H,W] tensor")
        P, H, W = src.shape
        if tuple(guide.shape) != (H, W):
            raise DvcError("fgs_filter: guide and planes differ in size")
        guide = guide.contiguous()
        out = torch.empty_like(src)
        self._check(self.lib.dvc_fgs_filter(self.h, ctypes.c_void_p(guide.data_ptr()), _ptr(src), P, H, W, float(lam), float(sigma_color),
                                            float(lambda_attenuation), int(num_iter), _ptr(out), _stream(src.device)), "dvc_fgs_filter")
        return out

    def l_to_guide8(self, l):
        """uint8(uncenter_l(L) * 255 / 100) (test.py:106) for a CUDA float32 [H,W] centred-luminance plane."""
        l = _dev_f32(l, "l_to_guide8 input")
        H, W = l.shape[-2:]
        out = torch.empty(H, W, device=l.device, dtype=torch.uint8)
        self._check(self.lib.dvc_l_to_guide8(self.h, _ptr(l), H, W, ctypes.c_void_p(out.data_ptr()), _stream(l.device)), "dvc_l_to_guide8")
        return out

    def centerpad_rgb8(self, rgb, size):
        """CenterPad(size) + CenterCrop(size) of test.py:44-46 for a CUDA uint8 [H,W,3] image -> uint8 [size[0],size[1],3]."""
        from dvc.prepost import centerpad_geometry

        if not (isinstance(rgb, torch.Tensor) and rgb.is_cuda and rgb.dtype == torch.uint8 and rgb.dim() == 3 and rgb.shape[2] == 3):
            raise DvcError("centerpad_rgb8: expected a CUDA uint8 tensor [H,W,3]")
        rgb = rgb.contiguous()
        Hs, Ws, _ = rgb.shape
        Hr, Wr, oy, ox = centerpad_geometry(Hs, Ws, size)
        out = torch.empty(size[0], size[1], 3, device=rgb.device, dtype=torch.uint8)
        self._check(self.lib.dvc_resize_antialias_crop_rgb8(self.h, ctypes.c_void_p(rgb.data_ptr()), Hs, Ws, Hr, Wr, oy, ox,
                                                            ctypes.c_void_p(out.data_ptr()), size[0], size[1], _stream(rgb.device)),
                    "dvc_resize_antialias_crop_rgb8")
        return out

    # ---- whole frames in, whole frames out -------------------------------------------------------------
    @staticmethod
    def _geometry(Hs, Ws, size):
        from dvc.prepost import centerpad_geometry

        Ho, Wo = int(size[0]), int(size[1])
        if Ho % 2 or Wo % 2:
            raise DvcError("the output size must be even (the networks run at half of it)")
        return centerpad_geometry(Hs, Ws, (Ho, Wo)) + (Ho, Wo)

    def ingest_rgb8(self, frames, size):
        """test.py:44-46,71 for CUDA uint8 frames [F,Hs,Ws,3]: CenterPad + CenterCrop to `size`, Lab, centred L only ->
        (L [F,1,Ho,Wo], L at half size [F,1,Ho/2,Wo/2]).  Equals centerpad_rgb8 -> rgb8_to_lab -> [:, 0:1] -> resize_half."""
        if not (isinstance(frames, torch.Tensor) and frames.is_cuda and frames.dtype == torch.uint8 and frames.dim() == 4
                and frames.shape[3] == 3):
            raise DvcError("ingest_rgb8: expected a CUDA uint8 tensor [F,H,W,3]")
        frames = frames.contiguous()
        F_, Hs, Ws, _ = frames.shape
        Hr, Wr, oy, ox, Ho, Wo = self._geometry(Hs, Ws, size)
        l = torch.empty(F_, 1, Ho, Wo, device=frames.device, dtype=torch.float32)
        lh = torch.empty(F_, 1, Ho // 2, Wo // 2, device=frames.device, dtype=torch.float32)
        self._check(self.lib.dvc_ingest_rgb8(self.h, ctypes.c_void_p(frames.data_ptr()), F_, Hs, Ws, Hr, Wr, oy, ox, Ho, Wo, _ptr(l),
                                             _ptr(lh), _stream(frames.device)), "dvc_ingest_rgb8")
        return l, lh

    def postprocess_rgb8(self, l, ab_half, wls=True, lam=500.0, sigma_color=4.0):
        """test.py:99-119 for CUDA l [F,1,Ho,Wo] (centred) and ab_half [F,2,Ho/2,Wo/2]: x2 * 1.25, the WLS filter guided by
        each frame's own L (when wls), Lab -> sRGB uint8 [F,Ho,Wo,3]."""
        l, ab_half = _dev_f32(l, "postprocess_rgb8 l"), _dev_f32(ab_half, "postprocess_rgb8 ab")
        F_, c1, Ho, Wo = l.shape
        if c1 != 1 or tuple(ab_half.shape) != (F_, 2, Ho // 2, Wo // 2):
            raise DvcError("postprocess_rgb8: expected l [F,1,Ho,Wo] and ab [F,2,Ho/2,Wo/2]")
        out = torch.empty(F_, Ho, Wo, 3, device=l.device, dtype=torch.uint8)
        self._check(self.lib.dvc_postprocess_rgb8(self.h, _ptr(l), _ptr(ab_half), F_, Ho, Wo, 1 if wls else 0, float(lam),
                                                  float(sigma_color), ctypes.c_void_p(out.data_ptr()), _stream(l.device)),
                    "dvc_postprocess_rgb8")
        return out

    def colorize_video_rgb8(self, frames, size, temperature=1e-10, wls=True, lam=500.0, sigma_color=4.0, continue_clip=False,
                            out=None):
        """K frames of a clip, uint8 sRGB [K,Hs,Ws,3] -> colourised uint8 sRGB [K,size[0],size[1],3] (test.py:29-125 without
        the file I/O), against the exemplar of set_exemplar, which must be size / 2.  continue_clip=True continues the
        recurrence from the last frame of the previous call.  `frames` may be a (preferably pinned) CPU tensor or a CUDA
        tensor; `out` lives where `frames` lives."""
        if not (isinstance(frames, torch.Tensor) and frames.dtype == torch.uint8 and frames.dim() == 4 and frames.shape[3] == 3):
            raise DvcError("colorize_video_rgb8 takes a uint8 tensor [K,H,W,3]")
        if frames.shape[0] < 1:
            raise DvcError("colorize_video_rgb8: no frames")
        frames = frames.contiguous()
        K, Hs, Ws, _ = frames.shape
        Hr, Wr, oy, ox, Ho, Wo = self._geometry(Hs, Ws, size)
        if out is None:
            out = torch.empty(K, Ho, Wo, 3, dtype=torch.uint8, device=frames.device)
            if not frames.is_cuda:
                out = out.pin_memory()
        if (out.is_cuda != frames.is_cuda or out.dtype != torch.uint8 or not out.is_contiguous()
                or tuple(out.shape) != (K, Ho, Wo, 3)):
            raise DvcError("colorize_video_rgb8: `out` must be a contiguous uint8 [K,Ho,Wo,3] tensor on the same side as the frames")
        rc = self.lib.dvc_colorize_video_rgb8(self.h, ctypes.c_void_p(frames.data_ptr()), K, Hs, Ws, Hr, Wr, oy, ox, Ho, Wo,
                                              float(temperature), 1 if wls else 0, float(lam), float(sigma_color),
                                              1 if continue_clip else 0, ctypes.c_void_p(out.data_ptr()), _stream(self.device))
        self._check(rc, "dvc_colorize_video_rgb8")
        return out

    # ---- query-row-sharded correlation: peer-mapped result buffers (CUDA IPC) ----------------------------
    def peer_buffer_create(self, nbytes):
        """(device pointer, 64-byte IPC handle) of a fresh zeroed cudaMalloc allocation other ranks can map."""
        ptr, handle = ctypes.c_void_p(0), ctypes.create_string_buffer(64)
        self._check(self.lib.dvc_peer_buffer_create(self.h, int(nbytes), ctypes.byref(ptr), handle), "dvc_peer_buffer_create")
        return ptr.value, handle.raw

    def peer_buffer_open(self, handle):
        ptr = ctypes.c_void_p(0)
        self._check(self.lib.dvc_peer_buffer_open(self.h, ctypes.create_string_buffer(bytes(handle), 64), ctypes.byref(ptr)),
                    "dvc_peer_buffer_open")
        return ptr.value

    def peer_buffer_close(self, ptr):
        self._check(self.lib.dvc_peer_buffer_close(self.h, ctypes.c_void_p(ptr)), "dvc_peer_buffer_close")

    def peer_buffer_destroy(self, ptr):
        self._check(self.lib.dvc_peer_buffer_destroy(self.h, ctypes.c_void_p(ptr)), "dvc_peer_buffer_destroy")

    def corr_set_peer_outputs(self, y4_ptrs=(), sim_ptrs=(), row0=0):
        """Route the result rows of the next corr_softmax_warp calls into these peer buffers as well (empty = off)."""
        n = len(y4_ptrs)
        ya = (ctypes.c_void_p * max(n, 1))(*[ctypes.c_void_p(p) for p in y4_ptrs])
        sa = (ctypes.c_void_p * max(n, 1))(*[ctypes.c_void_p(p) for p in sim_ptrs])
        self._check(self.lib.dvc_corr_set_peer_outputs(self.h, n, ya, sa, int(row0)), "dvc_corr_set_peer_outputs")

    def raw_view(self, ptr, numel):
        """float32 tensor view of `numel` elements at a device pointer owned by the library."""
        return _raw_view(ptr, numel, self.device)

    # ---- multi-GPU: exemplar operands as one flat buffer (broadcast with torch.distributed / NCCL) ----
    def exemplar_pack_size(self, H, W):
        return int(self.lib.dvc_exemplar_pack_size(self.h, H, W))

    def exemplar_export(self, H, W):
        buf = torch.empty(self.exemplar_pack_size(H, W), device=self.device, dtype=torch.float32)
        self._check(self.lib.dvc_exemplar_export(self.h, _ptr(buf), buf.numel(), _stream(self.device)),
                    "dvc_exemplar_export")
        return buf

    def exemplar_import(self, buf, H, W):
        buf = _dev_f32(buf, "exemplar pack")
        self._check(self.lib.dvc_exemplar_import(self.h, _ptr(buf), buf.numel(), H, W, _stream(self.device)),
                    "dvc_exemplar_import")

    # ---- debug hooks ---------------------------------------------------------------------------------
    def debug_flag(self, name, value):
        self._check(self.lib.dvc_debug_set_flag(self.h, name.encode(), int(value)), "dvc_debug_set_flag")

    def debug_conv2d(self, net, name, x, cout, dil=1, stride=1, act=0, slope=0.0, reflect=False, upconv=False,
                     fuse_tail=False, in_bound=None, out_planes=False, add=None, want_stats=False):
        """One convolution layer (weights `name` of `net`) on a CUDA NCHW tensor through the engine the layer programs
        use (include/dvc.h: dvc_debug_conv2d).  Returns y or (y, stats [B,cout,2] float64)."""
        x = _dev_f32(x, "debug_conv2d input")
        B, _, H, W = x.shape
        Ho, Wo = (2 * H, 2 * W) if upconv else ((H + stride - 1) // stride, (W + stride - 1) // stride)
        y = torch.empty(B, 2 if fuse_tail else cout, Ho, Wo, device=x.device, dtype=torch.float32)
        st = torch.zeros(B, cout, 2, device=x.device, dtype=torch.float64) if want_stats else None
        bound = float(x.abs().max()) if in_bound is None else float(in_bound)
        add = _dev_f32(add, "debug_conv2d addend") if add is not None else None
        rc = self.lib.dvc_debug_conv2d(self.h, net, name.encode(), _ptr(x), B, H, W, dil, stride, act, float(slope),
                                       1 if reflect else 0, 1 if upconv else 0, 1 if fuse_tail else 0, bound,
                                       1 if out_planes else 0, _ptr(add), _ptr(y), _ptr(st), _stream(x.device))
        self._check(rc, "dvc_debug_conv2d")
        return (y, st) if want_stats else y

    def debug_buffer(self, name, act=True):
        """Copy of an internal workspace.  act=True: padded NHWC activation -> interior as NCHW [B,C,H,W]."""
        ptr, nbytes, sig = ctypes.c_void_p(0), ctypes.c_int64(0), (ctypes.c_int * 5)()
        self._check(self.lib.dvc_debug_get_buffer(self.h, name.encode(), ctypes.byref(ptr), ctypes.byref(nbytes), sig),
                    "dvc_debug_get_buffer")
        torch.cuda.synchronize(self.device)
        flat = _raw_view(ptr.value, nbytes.value // 4, self.device).clone()
        if not act:
            return flat
        B, H, W, C, P = list(sig)
        split = P < 0  # hi/lo planes of a tensor-core activation are stored back to back
        if split:
            P = -1 - P
        mode16, P = divmod(P, 1000)  # 2: fp16 hi/lo planes of value * 2^e only; 3: an fp32 plane followed by them
        n = B * (H + 2 * P) * (W + 2 * P) * C
        if mode16 == 2:
            # the static exponent lives in the layer program; return hi + lo in scaled units
            halves = flat.view(torch.float16)
            t = halves[:n].float() + halves[n:2 * n].float()
        else:
            t = flat[:n] + flat[n:2 * n] if split else flat[:n]
        t = t.view(B, H + 2 * P, W + 2 * P, C)
        return t[:, P:P + H, P:P + W, :].permute(0, 3, 1, 2).contiguous()

    # ---- introspection ---------------------------------------------------------------------------
    def launch_count(self, reset=False):
        return int(self.lib.dvc_launch_count(self.h, 1 if reset else 0))

    def profile_corr(self, enable=True):
        self._check(self.lib.dvc_profile_corr(self.h, 1 if enable else 0), "dvc_profile_corr")

    def profile_conv(self, enable=True):
        self._check(self.lib.dvc_profile_conv(self.h, 1 if enable else 0), "dvc_profile_conv")

    def conv_profile(self, variant=0, reset=False):
        """(launches, total ms, total algorithmic FLOPs) of the recorded tensor-core conv launches of `variant`."""
        ms, fl = ctypes.c_double(0), ctypes.c_double(0)
        n = self.lib.dvc_conv_profile(self.h, variant, 1 if reset else 0, ctypes.byref(ms), ctypes.byref(fl))
        return int(n), ms.value, fl.value

    def corr_mean_ms(self, reset=True):
        return float(self.lib.dvc_corr_mean_ms(self.h, 1 if reset else 0))


def _raw_view(ptr, n_floats, device):
    """float32 tensor aliasing raw device memory (debug only) via the CUDA array interface."""

    class _Holder:
        pass

    h = _Holder()
    h.__cuda_array_interface__ = {"shape": (n_floats,), "typestr": "<f4", "data": (ptr, False), "version": 2}
    return torch.as_tensor(h, device=device)


_contexts = {}


def get_context(device=None):
    """Process-wide context of a device (shared by the three drop-in modules, like test.py:147-166)."""
    if device is None:
        device = torch.cuda.current_device() if torch.cuda.is_available() else 0
    idx = device if isinstance(device, int) else (torch.device(device).index or 0)
    if idx not in _contexts:
        _contexts[idx] = Context(idx)
    return _contexts[idx]
