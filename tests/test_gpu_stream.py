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
    """tools/colorize_folder.py's data flow before it streamed: every frame decoded up front, every step over the clip.
    `frames` is a uint8 [F,H,W,3] tensor or a list of uint8 [H,W,3] frames whose sizes may differ (each is CenterPad-ed
    to `size` on its own)."""
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


@pytest.fixture
def flags(ctx):
    """ctx.debug_flag for one test; the shipped values come back afterwards, also when the test fails."""
    yield ctx.debug_flag
    ctx.debug_flag("video_batch", 8)
    ctx.debug_flag("clip_astreams", 1)


def video_calls(ctx, frames, sizes, wls=True):
    """The clip in consecutive calls of `sizes` frames, the recurrence continued across them."""
    pinned, out, t = frames.pin_memory(), [], 0
    for k in sizes:
        out.append(ctx.colorize_video_rgb8(pinned[t:t + k], SIZE, wls=wls, continue_clip=t > 0))
        t += k
    assert t == len(frames)
    return torch.cat(out)


@pytest.mark.parametrize("wls", [True, False])
@pytest.mark.parametrize("K", [1, 4, 11])
@pytest.mark.parametrize("G", [1, 3, 8])
def test_streamed_chunks_equal_composition(ctx, flags, clip11, G, K, wls):
    """G frames per post-processing batch: batch b uses half b & 1 of the L and ab rings, so G = 1 and 3 wrap them several
    times inside one call, G = 3 with K = 11 ends in a partial batch of 2 after a wrap, and K = 4 with G = 3 puts call
    boundaries in the middle of a batch."""
    frames, ref = clip11
    want = composition(ctx, frames, ref, SIZE, wls)  # also installs the exemplar
    flags("video_batch", G)
    got = video_calls(ctx, frames, [min(K, 11 - t) for t in range(0, 11, K)], wls)
    assert torch.equal(got, want)


@pytest.fixture(scope="module")
def clip40():
    return seeded_frames(41, 40, 90, 120), seeded_frames(42, 1, 90, 120)[0]


@pytest.mark.parametrize("wls", [True, False])
@pytest.mark.parametrize("sizes,astreams", [((40,), 1), ((17, 23), 1), ((37, 3), 1), ((17, 23), 2)])
def test_video_rings_wrap_at_the_default_batch(ctx, flags, clip40, sizes, astreams, wls):
    """The shipped G = 8 past 2G frames in one call, where ingest and ColorVidNet wait for batch b - 2's post-processing
    before they reuse its ring slots: 40 frames are five batches (the rings wrap twice, the last batch is full); 17 + 23
    and 37 + 3 put the call boundary in the middle of a batch.  clip_astreams = 2 has frames t+1 and t+2 in flight on two
    phase-A streams."""
    frames, ref = clip40
    want = composition(ctx, frames, ref, SIZE, wls)
    flags("clip_astreams", astreams)
    assert torch.equal(video_calls(ctx, frames, sizes, wls), want)


def test_source_size_changes_mid_clip(ctx, clip11):
    """Runs of 90 x 120, 150 x 180, 90 x 120 and 100 x 300 frames, each longer than 2G: the source frame and the ingest work
    buffers regrow in the middle of a continued clip.  Once with one call per run, once through colorize_stream, which
    ends a chunk at each size change."""
    _, ref = clip11
    runs = [seeded_frames(50 + i, n, h, w) for i, (n, h, w) in enumerate([(18, 90, 120), (22, 150, 180), (19, 90, 120), (18, 100, 300)])]
    frames = [f for run in runs for f in run]
    want = composition(ctx, frames, ref, SIZE)
    got = torch.cat([ctx.colorize_video_rgb8(run.pin_memory(), SIZE, continue_clip=i > 0) for i, run in enumerate(runs)])
    assert torch.equal(got, want)
    streamed = list(colorize_stream(ctx, iter([f.numpy() for f in frames]), ref.numpy(), SIZE, chunk=20, workers=2))
    assert torch.equal(torch.from_numpy(np.stack(streamed)), want)


def test_product_geometry(ctx):
    """The geometry of profiles/stream_bench.json: 1080 x 1920 sources at image_size 960 x 1728 (the nets at 480 x 864), 20
    frames in one call with the WLS filter: rings at full size, FGS batched over 8 frames of 960 x 1728."""
    frames = torch.cat([seeded_frames(61 + t, 1, 1080, 1920) for t in range(20)])  # 124 MB; one frame of noise at a time
    ref = seeded_frames(62, 1, 1080, 1920)[0]
    size = (960, 1728)
    want = composition(ctx, frames, ref, size)
    got = ctx.colorize_video_rgb8(frames.pin_memory(), size, continue_clip=False)
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
