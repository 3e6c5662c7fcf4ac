"""GPU: the pre / post-processing kernels of the streaming path against the CPU oracle, at the shapes and edges the video
driver runs at.  The FGS kernels were written to the oracle's operation order and are held to it bit for bit; the
frame-batched ingest and post-processing are held to the oracle within the float64-vs-fp32 and pow() caveats that
tests/test_gpu_prepost.py documents."""
import numpy as np
import pytest
import torch

from oracle import dvc_oracle as O
from oracle import prepost_oracle as P
from test_gpu_stream import seeded_frames

pytestmark = pytest.mark.gpu

L_TOL = 7.7e-6  # one fp32 ulp at |L| = 100 (the float64 Lab is rounded to fp32 before L - 50 on both sides)


# ------------------------------------------------------------------------------------------------ B1: FGS bit for bit
def _zigzag():
    """0, 255, 1, 254, ..., 127, 128, 128: consecutive differences 255, 254, ..., 1, 0."""
    s = np.empty(257, np.int64)
    s[0:256:2], s[1:256:2], s[256] = np.arange(128), 255 - np.arange(128), 128
    return s


def make_guide(kind, H, W, seed):
    i, j = np.meshgrid(np.arange(H), np.arange(W), indexing="ij")
    if kind == "random":
        return np.random.default_rng(seed).integers(0, 256, (H, W)).astype(np.uint8)
    if kind == "flat":  # every weight is the LUT's d = 0 entry
        return np.full((H, W), 117, np.uint8)
    if kind == "stripes":  # hard 0 / 255 edges along both axes
        return (255 * (((i // 3) + (j // 2)) & 1)).astype(np.uint8)
    if kind == "lut":  # horizontal and vertical neighbours differ by every d in 0..255 once H + W > 257
        return _zigzag()[(i + j) % 257].astype(np.uint8)
    raise ValueError(kind)


FGS_SHAPES = [(2, 2), (2, 97), (97, 2), (31, 33), (32, 32), (33, 65), (64, 31), (100, 129), (432, 768)]
# (lambda, sigma_color, lambda_attenuation, num_iter); sigma 0.5 puts fp32 subnormals into the LUT (d = 44..51)
FGS_PARAMS = [(500.0, 4.0, 0.25, 3), (0.0, 4.0, 0.25, 3), (1e4, 0.5, 0.25, 3), (500.0, 4.0, 0.5, 1), (500.0, 4.0, 0.25, 5)]


@pytest.mark.parametrize("lam,sigma,att,iters", FGS_PARAMS)
@pytest.mark.parametrize("kind", ["random", "flat", "stripes", "lut"])
@pytest.mark.parametrize("planes", [1, 3])
@pytest.mark.parametrize("H,W", FGS_SHAPES)
def test_fgs_filter_bit_exact(ctx, H, W, planes, kind, lam, sigma, att, iters):
    """The horizontal sweep's 32 x 32 shared-memory tiles at widths and heights that are not multiples of 32, and one-row
    / one-column tiles, against oracle/prepost_oracle.py: the same separately rounded fp32 operations in the same order,
    so the same bits."""
    guide = make_guide(kind, H, W, H * 1000 + W)
    src = (np.random.default_rng(H + 7 * W + planes).standard_normal((planes, H, W)) * 30).astype(np.float32)
    out = ctx.fgs_filter(torch.from_numpy(guide).cuda(), torch.from_numpy(src).cuda(), lam, sigma, att, iters).cpu().numpy()
    ref = P.fgs_filter(guide, src, lam, sigma, att, iters)
    assert np.array_equal(out, ref), (np.abs(out - ref).max(), int((out != ref).sum()))


@pytest.mark.parametrize("H,W", FGS_SHAPES)
def test_l_to_guide8_bit_exact(ctx, H, W):
    """Random L over and beyond [-50, 50] (the clamps), with the values where (L + 50) * 255 / 100 is an integer (where
    the truncation flips) placed first."""
    l = np.random.default_rng(H * W).uniform(-55.0, 55.0, (H, W)).astype(np.float32)
    edges = np.float32(np.arange(256) * 100.0 / 255.0 - 50.0)
    n = min(l.size, edges.size)
    l.reshape(-1)[:n] = edges[:n]
    out = ctx.l_to_guide8(torch.from_numpy(l).cuda()).cpu().numpy()
    assert np.array_equal(out, P.l_to_guide8(l))


# ------------------------------------------------------------------------------------------------ B2: postprocess_rgb8
def _assert_rgb8_close(out, ref):
    """One level on at most 1e-5 of the values: CUDA's and numpy's double pow() may differ in the last ulp, which flips a
    truncation only where v * 255 sits within ~1e-13 of an integer (test_lab_to_rgb8_matches_float64_oracle)."""
    assert out.shape == ref.shape and out.dtype == ref.dtype == torch.uint8
    d = (out.int() - ref.int()).abs()
    assert int(d.max()) <= 1 and float((d > 0).float().mean()) <= 1e-5, (int(d.max()), int((d > 0).sum()))


@pytest.mark.parametrize("wls", [True, False])
@pytest.mark.parametrize("F,size", [(8, (64, 96)), (8, (70, 98)), (2, (432, 768)), (1, (2, 2))])
def test_postprocess_rgb8_vs_oracle(ctx, F, size, wls):
    """ab on a 1/8 grid with |ab| <= 100: the bilinear x2 weights (0.25, 0.75) and the factor 1.25 round nowhere, so the
    up-sampled ab is exact on both sides and the rest of the chain is held to the oracle."""
    g = torch.Generator().manual_seed(F * 1000 + size[0])
    l = torch.rand(F, 1, *size, generator=g) * 100 - 50
    ab = torch.randint(-800, 801, (F, 2, size[0] // 2, size[1] // 2), generator=g).float() / 8
    up_ref = O.upsample2_scaled(ab)
    assert torch.equal(ctx.upsample2_scaled(ab.cuda()).cpu(), up_ref)  # the premise of this test
    out = ctx.postprocess_rgb8(l.cuda(), ab.cuda(), wls=wls).cpu()
    ref = []
    for t in range(F):
        up = up_ref[t].numpy()
        if wls:
            up = P.fgs_filter(P.l_to_guide8(l[t, 0].numpy()), up, 500.0, 4.0)
        ref.append(O.lab_to_rgb8(l[t:t + 1], torch.from_numpy(np.ascontiguousarray(up))[None]))
    _assert_rgb8_close(out, torch.cat(ref))


# ------------------------------------------------------------------------------------------------ B3: ingest_rgb8
@pytest.mark.parametrize("hs,ws,size", [
    (1080, 1920, (960, 1728)),  # resized to 972 x 1728, 6 rows cropped; sigma 0.056: a one-tap Gaussian
    (1080, 1920, (432, 768)),   # same aspect ratio; sigma 0.75, radius 3
    (1920, 1080, (432, 768)),   # portrait: resized to 1365 x 768, 466 rows cropped
    (90, 120, (64, 96)),        # the clip of test_gpu_stream.py
    (27, 48, (64, 96)),         # up-scaled to 64 x 113, 8 columns cropped
    (1, 200, (64, 96)),         # one source row (mirror_idx with n = 1), up-scaled to 64 x 12800
    (200, 1, (64, 96)),         # one source column, up-scaled to 19200 x 96
])
def test_ingest_rgb8_vs_oracle(ctx, hs, ws, size):
    F = 3
    frames = seeded_frames(hs * 7 + ws, F, hs, ws)
    l, lh = ctx.ingest_rgb8(frames.cuda(), size)
    l, lh = l.cpu(), lh.cpu()
    ref = torch.cat([O.rgb8_to_lab(torch.from_numpy(P.centerpad_transform(f.numpy(), size))[None])[:, 0:1] for f in frames])
    assert l.shape == ref.shape == (F, 1) + tuple(size)
    # a uint8 pixel that truncates the other way on one side changes L by far more than an ulp (test_centerpad_resize_vs_scipy)
    flipped = (l - ref).abs() > L_TOL
    assert float(flipped.float().mean()) <= 1e-5, int(flipped.sum())
    ref_half = O.resize_half(ref)
    clean = ~flipped.view(F, 1, size[0] // 2, 2, size[1] // 2, 2).any(5).any(3)
    assert lh.shape == ref_half.shape
    assert float((lh - ref_half).abs()[clean].max()) <= 1e-5


# ------------------------------------------------------------------------------------------------ B4: the whole 8-bit cube
def test_colour_conversions_over_the_whole_cube(ctx):
    """rgb8_to_lab on all 2^24 colours (one 4096 x 4096 image) against the float64 oracle, then the round trip through
    lab_to_rgb8 within one level (truncating output conversion)."""
    idx = torch.arange(1 << 24, dtype=torch.int64)
    rgb = torch.stack([(idx >> 16) & 255, (idx >> 8) & 255, idx & 255], -1).to(torch.uint8).view(1, 4096, 4096, 3)
    lab_dev = ctx.rgb8_to_lab(rgb.cuda())
    lab = lab_dev.cpu().numpy()
    differ, worst = 0, [0.0, 0.0, 0.0]
    for r0 in range(0, 4096, 512):
        ref = O.rgb8_to_lab(rgb[:, r0:r0 + 512]).numpy()
        out = lab[:, :, r0:r0 + 512]
        differ += int((out != ref).sum())
        dl = np.abs(out[:, 0] - ref[:, 0])
        assert dl.max() <= L_TOL, (r0, dl.max())
        worst[0] = max(worst[0], float(dl.max()))
        for c in (1, 2):  # a, b: one fp32 ulp of the value
            d = np.abs(out[:, c] - ref[:, c])
            ulps = d / np.spacing(np.abs(ref[:, c]))
            assert ulps.max() <= 1.0, (r0, c, float(ulps.max()), float(ref[:, c].reshape(-1)[ulps.argmax()]))
            worst[c] = max(worst[c], float(ulps.max()))
    print(f"\nrgb8_to_lab over 2^24 colours: {differ} of {3 << 24} values not identical to the oracle; "
          f"max |dL| = {worst[0]:.3g}, max |da|, |db| = {worst[1]:.3g}, {worst[2]:.3g} ulp")
    back = ctx.lab_to_rgb8(lab_dev[:, 0:1].contiguous(), lab_dev[:, 1:3].contiguous())
    assert int((back.int() - rgb.cuda().int()).abs().max()) <= 1


# ------------------------------------------------------------------------------------------------ B5: lab_to_rgb8 branches
T_F = 0.2068966  # lab2xyz: cube above, linear segment below
T_GAMMA = 0.0031308  # xyz2rgb: gamma above, linear segment below


def _ladder(v, n=8):
    """fp32 values from n ulps below to n ulps above v."""
    v = np.float32(v)
    down, up = [v], [v]
    for _ in range(n):
        down.append(np.nextafter(down[-1], np.float32(-np.inf)))
        up.append(np.nextafter(up[-1], np.float32(np.inf)))
    return np.array(down[::-1] + up[1:], np.float32)


def _linear_rgb(L, a, b):
    """The oracle's lab2rgb up to the gamma step, float64: linear sRGB [..., 3] of centred L."""
    y = (L.astype(np.float64) + 66.0) / 116.0
    f = np.stack([a / 500.0 + y, y, np.maximum(y - b / 200.0, 0.0)], -1)
    xyz = np.where(f > T_F, f ** 3, (f - 16.0 / 116.0) / 7.787) * np.array([0.95047, 1.0, 1.08883])
    M = np.array([[0.412453, 0.357580, 0.180423], [0.212671, 0.715160, 0.072169], [0.019334, 0.119193, 0.950227]])
    return xyz @ np.linalg.inv(M).T


def lab_branch_grid():
    """(L, a, b) samples: a coarse grid over and beyond the gamut (clipping to 0 and 1, a, b at +-128), plus fp32 ladders
    across f = 0.2068966 on each of x, y, z, across z = 0 (large positive b) and across the 0.0031308 gamma knee of each
    output channel."""
    pts = []
    Lg, ag = np.linspace(-52, 52, 53, dtype=np.float32), np.linspace(-128, 128, 33, dtype=np.float32)
    pts.append(np.stack(np.meshgrid(Lg, ag, ag, indexing="ij"), -1).reshape(-1, 3))
    others = np.array([-128, -40, 0, 40, 128], np.float32)
    Ls = np.linspace(-50, 50, 41)
    fy = (Ls + 66.0) / 116.0
    # y: L + 50 = 116 f - 16 (L ~ -42)
    L_y = _ladder(116.0 * T_F - 66.0)
    pts.append(np.stack(np.meshgrid(L_y, others, others, indexing="ij"), -1).reshape(-1, 3))
    for L, f in zip(Ls, fy):
        for v, col in ((500.0 * (T_F - f), 1), (200.0 * (f - T_F), 2), (200.0 * f, 2)):  # x, z at the knee; z = 0
            if abs(v) > 128:
                continue
            lad = _ladder(v)
            for o in others:
                s = np.empty((lad.size, 3), np.float32)
                s[:, 0], s[:, col], s[:, 3 - col] = L, lad, o
                pts.append(s)
    # the gamma knee: for each (a, b) and output channel, the L where linear sRGB crosses 0.0031308 (bisection in float64)
    for a in (-20.0, 0.0, 20.0):
        for b in (-20.0, 0.0, 20.0):
            for k in range(3):
                lo, hi = -50.0, 0.0
                g = lambda L: _linear_rgb(np.array([L]), a, b)[0, k] - T_GAMMA  # noqa: E731
                if g(lo) > 0 or g(hi) < 0:
                    continue
                for _ in range(80):
                    mid = 0.5 * (lo + hi)
                    lo, hi = (mid, hi) if g(mid) < 0 else (lo, mid)
                lad = _ladder(lo, 16)
                pts.append(np.stack([lad, np.full_like(lad, a), np.full_like(lad, b)], -1))
    return np.concatenate(pts)


def test_lab_to_rgb8_branches_vs_oracle(ctx):
    lab = lab_branch_grid()
    n = lab.shape[0]
    l = torch.from_numpy(np.ascontiguousarray(lab[:, 0])).view(1, 1, 1, n)
    ab = torch.from_numpy(np.ascontiguousarray(lab[:, 1:].T)).view(1, 2, 1, n)
    out = ctx.lab_to_rgb8(l.cuda(), ab.cuda()).cpu()
    _assert_rgb8_close(out, O.lab_to_rgb8(l, ab))
