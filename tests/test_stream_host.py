"""CPU: the host side of dvc/stream.py (decode pool, chunking, order, error hand-over) against a fake context that
records its calls and "colourises" a frame by resizing it with nearest neighbours."""
import threading

import numpy as np
import pytest
import torch

from dvc.stream import colorize_stream


class FakeContext:
    device = torch.device("cpu")

    def __init__(self, fail_at_call=None):
        self.calls, self.exemplar, self.fail_at_call = [], None, fail_at_call
        self.lock = threading.Lock()

    # exemplar path: centerpad_rgb8 -> rgb8_to_lab -> resize_half -> set_exemplar
    def centerpad_rgb8(self, rgb, size):
        return rgb[: size[0], : size[1]]

    def rgb8_to_lab(self, rgb):
        return rgb.permute(0, 3, 1, 2).float()

    def resize_half(self, x):
        return x[:, :, ::2, ::2]

    def set_exemplar(self, lab):
        self.exemplar = tuple(lab.shape)

    def colorize_video_rgb8(self, frames, size, temperature, wls, lam, sigma_color, continue_clip=False, out=None):
        with self.lock:
            self.calls.append((tuple(frames.shape), continue_clip))
            if self.fail_at_call is not None and len(self.calls) == self.fail_at_call:
                raise RuntimeError("device failure")
        K, Hs, Ws, _ = frames.shape
        ys = torch.arange(size[0]) * Hs // size[0]
        xs = torch.arange(size[1]) * Ws // size[1]
        out.copy_(frames[:, ys][:, :, xs])
        return out


def make_frame(i, h=6, w=10):
    return np.full((h, w, 3), i % 251, np.uint8) + np.arange(w, dtype=np.uint8)[None, :, None]


def expected(frame, size):
    ys = np.arange(size[0]) * frame.shape[0] // size[0]
    xs = np.arange(size[1]) * frame.shape[1] // size[1]
    return frame[ys][:, xs]


SIZE = (4, 8)
EX = np.zeros((6, 10, 3), np.uint8)


def test_order_and_short_last_chunk():
    ctx = FakeContext()
    frames = [make_frame(i) for i in range(11)]
    out = list(colorize_stream(ctx, iter(frames), EX, SIZE, chunk=4, workers=3))
    assert len(out) == 11
    for f, o in zip(frames, out):
        assert o.shape == (4, 8, 3) and o.dtype == np.uint8
        assert np.array_equal(o, expected(f, SIZE))
    assert [c[0][0] for c in ctx.calls] == [4, 4, 3]  # the last chunk is shorter
    assert [c[1] for c in ctx.calls] == [False, True, True]  # one clip: only the first call starts from zeros
    assert ctx.exemplar == (1, 3, 2, 4)


def test_decode_runs_on_the_pool_and_keeps_order():
    ctx = FakeContext()
    seen = set()

    def decode(i):
        seen.add(threading.get_ident())
        return make_frame(i)

    out = list(colorize_stream(ctx, range(9), EX, SIZE, decode=decode, chunk=2, workers=4))
    assert [int(o[0, 0, 0]) for o in out] == [expected(make_frame(i), SIZE)[0, 0, 0] for i in range(9)]
    assert threading.get_ident() not in seen


def test_source_size_change_ends_the_chunk():
    ctx = FakeContext()
    frames = [make_frame(i) for i in range(3)] + [make_frame(i, 12, 20) for i in range(3, 5)] + [make_frame(5)]
    out = list(colorize_stream(ctx, frames, EX, SIZE, chunk=8, workers=2))
    assert [c[0] for c in ctx.calls] == [(3, 6, 10, 3), (2, 12, 20, 3), (1, 6, 10, 3)]
    assert [c[1] for c in ctx.calls] == [False, True, True]  # the clip continues across the size change
    for f, o in zip(frames, out):
        assert np.array_equal(o, expected(f, SIZE))


def test_decode_exception_reaches_the_caller():
    def decode(i):
        if i == 5:
            raise ValueError("corrupt frame 5")
        return make_frame(i)

    got = []
    with pytest.raises(ValueError, match="corrupt frame 5"):
        for o in colorize_stream(FakeContext(), range(10), EX, SIZE, decode=decode, chunk=2, workers=2):
            got.append(o)
    assert len(got) == 4  # the two chunks before the failing one came out


def test_device_exception_reaches_the_caller():
    with pytest.raises(RuntimeError, match="device failure"):
        list(colorize_stream(FakeContext(fail_at_call=2), (make_frame(i) for i in range(8)), EX, SIZE, chunk=3))


def test_bad_frame_is_rejected():
    with pytest.raises(ValueError, match="uint8"):
        list(colorize_stream(FakeContext(), [np.zeros((6, 10), np.uint8)], EX, SIZE))


def test_early_close_stops_the_worker():
    before = threading.active_count()
    gen = colorize_stream(FakeContext(), (make_frame(i) for i in range(100)), EX, SIZE, chunk=2)
    next(gen)
    gen.close()
    assert threading.active_count() <= before
