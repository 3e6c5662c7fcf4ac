"""GPU: whole frames in, whole frames out -- dvc_ingest_rgb8, dvc_postprocess_rgb8 and dvc_colorize_video_rgb8 against the
composition of the existing per-step entry points, bit for bit, and the bounded device memory of a long stream."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import dvc
from dvc.stream import colorize_stream

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SIZE = (64, 96)  # the networks run at 32 x 48


def seeded_frames(seed, n, h, w):
    g = torch.Generator().manual_seed(seed)
    # blocky content + noise: edges and flats for the resize and the WLS filter
    base = torch.randint(0, 256, (n, h // 6 + 1, w // 6 + 1, 3), generator=g, dtype=torch.uint8)
    img = base.repeat_interleave(6, 1).repeat_interleave(6, 2)[:, :h, :w].int()
    return (img + torch.randint(-8, 9, img.shape, generator=g)).clamp(0, 255).to(torch.uint8)


def chain_ingest(ctx, frames, size):
    big = torch.stack([ctx.centerpad_rgb8(f, size) for f in frames])
    l = ctx.rgb8_to_lab(big)[:, 0:1].contiguous()
    return l, ctx.resize_half(l)


def chain_post(ctx, l, ab, wls, lam=500.0, sigma=4.0):
    up = ctx.upsample2_scaled(ab, 1.25)
    if wls:
        for t in range(up.shape[0]):
            up[t] = ctx.fgs_filter(ctx.l_to_guide8(l[t, 0]), up[t], lam, sigma)
    return ctx.lab_to_rgb8(l, up)


def composition(ctx, frames, ref, size, wls=True):
    """tools/colorize_folder.py's data flow before it streamed: every frame decoded up front, every step over the clip."""
    big = torch.stack([ctx.centerpad_rgb8(f.cuda(), size) for f in frames])
    lab_large = ctx.rgb8_to_lab(big)
    lab = ctx.resize_half(lab_large)
    ctx.set_exemplar(ctx.resize_half(ctx.rgb8_to_lab(ctx.centerpad_rgb8(ref.cuda(), size)[None])))
    ab = ctx.colorize_clip(lab[:, 0:1].contiguous(), 1e-10)
    ab_large = ctx.upsample2_scaled(ab, 1.25)
    if wls:
        for t in range(len(frames)):
            ab_large[t] = ctx.fgs_filter(ctx.l_to_guide8(lab_large[t, 0]), ab_large[t], 500.0, 4.0)
    return ctx.lab_to_rgb8(lab_large[:, 0:1].contiguous(), ab_large).cpu()


@pytest.mark.parametrize("hs,ws", [(150, 180), (100, 300), (96, 144), (40, 50)])
@pytest.mark.parametrize("F", [1, 3, 7])
def test_ingest_rgb8_equals_chain(ctx, hs, ws, F):
    """(150, 180): the taller branch of CenterPad (crop rows), (100, 300): the wider branch (crop columns), both down-scales
    with a non-trivial anti-aliasing Gaussian; (96, 144): same aspect; (40, 50): up-scale, no Gaussian."""
    frames = seeded_frames(hs * ws + F, F, hs, ws).cuda()
    l, lh = ctx.ingest_rgb8(frames, SIZE)
    rl, rlh = chain_ingest(ctx, frames, SIZE)
    assert l.shape == (F, 1) + SIZE and lh.shape == (F, 1, SIZE[0] // 2, SIZE[1] // 2)
    assert torch.equal(l, rl) and torch.equal(lh, rlh)


@pytest.mark.parametrize("size", [(64, 96), (38, 70)])
@pytest.mark.parametrize("wls", [True, False])
@pytest.mark.parametrize("F", [1, 5])
def test_postprocess_rgb8_equals_chain(ctx, size, wls, F):
    g = torch.Generator().manual_seed(F * 10 + size[0])
    l = (torch.rand(F, 1, *size, generator=g) * 100 - 50).cuda()
    ab = (torch.randn(F, 2, size[0] // 2, size[1] // 2, generator=g) * 40).cuda()
    out = ctx.postprocess_rgb8(l, ab, wls=wls)
    ref = chain_post(ctx, l, ab, wls)
    assert out.shape == (F,) + size + (3,) and out.dtype == torch.uint8
    assert torch.equal(out, ref)


@pytest.fixture(scope="module")
def clip11():
    frames = seeded_frames(21, 11, 90, 120)  # 90 x 120 -> 64 x 96: the crop branch, with a Gaussian on both axes
    ref = seeded_frames(22, 1, 90, 120)[0]
    return frames, ref


@pytest.mark.parametrize("wls", [True, False])
@pytest.mark.parametrize("K", [1, 4, 11])
def test_streamed_chunks_equal_composition(ctx, clip11, K, wls):
    frames, ref = clip11
    want = composition(ctx, frames, ref, SIZE, wls)  # also installs the exemplar
    pinned = frames.pin_memory()
    got = torch.cat([ctx.colorize_video_rgb8(pinned[t:t + K], SIZE, wls=wls, continue_clip=t > 0) for t in range(0, 11, K)])
    assert torch.equal(got, want)


def test_restart_mid_clip_and_stale_state(ctx, clip11):
    frames, ref = clip11
    want_tail = composition(ctx, frames[5:], ref, SIZE)
    ctx.colorize_video_rgb8(frames[:5], SIZE)
    tail = ctx.colorize_video_rgb8(frames[5:], SIZE, continue_clip=False)  # a fresh clip from here
    assert torch.equal(tail, want_tail)
    # a device-resident clip goes through the same path
    assert torch.equal(ctx.colorize_video_rgb8(frames[5:].cuda(), SIZE).cpu(), want_tail)
    ctx.colorize_video_rgb8(frames[:2], SIZE)
    ctx.set_exemplar(ctx.resize_half(ctx.rgb8_to_lab(ctx.centerpad_rgb8(ref.cuda(), SIZE)[None])))
    with pytest.raises(dvc.DvcError, match=r"\(-4\)"):  # DVC_ERR_STATE: the exemplar changed since
        ctx.colorize_video_rgb8(frames[2:4], SIZE, continue_clip=True)
    ctx.colorize_video_rgb8(frames[2:4], SIZE)
    with pytest.raises(dvc.DvcError, match=r"\(-2\)"):  # the nets' size must be the exemplar's
        ctx.colorize_video_rgb8(frames[2:4], (128, 192), continue_clip=True)


def test_device_memory_does_not_grow_with_the_clip(ctx, clip11):
    frames, ref = clip11
    src = seeded_frames(31, 96, 90, 120).numpy()
    chunk = 4

    def run(n):
        for _ in colorize_stream(ctx, iter(src[:n]), ref.numpy(), SIZE, chunk=chunk, workers=2):
            pass
        torch.cuda.synchronize()
        return torch.cuda.mem_get_info()[0]

    run(12)  # warm-up: every ring and workspace exists now
    free12 = run(12)
    free96 = run(96)
    # one chunk of frames in and out on the device, at least one 2 MB allocation granule
    slack = max(chunk * (90 * 120 * 3 + SIZE[0] * SIZE[1] * 3), 2 << 20)
    assert abs(free12 - free96) <= slack, (free12, free96)


def test_colorize_folder_tool_matches_composition(ctx, clip11, tmp_path):
    from PIL import Image

    frames, ref = clip11
    src, out = tmp_path / "frames", tmp_path / "out"
    src.mkdir()
    for i, f in enumerate(frames):
        Image.fromarray(f.numpy()).save(src / f"frame{i:03d}.png")
    Image.fromarray(ref.numpy()).save(tmp_path / "ref.png")
    subprocess.run([sys.executable, os.path.join(ROOT, "tools", "colorize_folder.py"), "--clip", str(src), "--ref",
                    str(tmp_path / "ref.png"), "--out", str(out), "--seeded-weights", "--image-size", str(SIZE[0]), str(SIZE[1])],
                   check=True, cwd=str(tmp_path))
    want = composition(ctx, frames, ref, SIZE)  # the tool's seeded weights are the suite's (dvc.synth, seed 0)
    for i in range(len(frames)):
        got = np.asarray(Image.open(out / f"frame{i:03d}.png"))
        assert np.array_equal(got, want[i].numpy()), i
