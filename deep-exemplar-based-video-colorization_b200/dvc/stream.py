"""Colourise a clip of any length, uint8 frames in and uint8 frames out, in bounded memory (test.py:29-125).

    for rgb in colorize_stream(ctx, paths, exemplar, (432, 768), decode=load_png):
        save(rgb)

A pool of decode threads runs ahead of the device; decoded frames are gathered into chunks of up to `chunk` frames in
one of two pinned host slots, each chunk goes through one Context.colorize_video_rgb8 call (the recurrence continues
across calls), and the colourised frames come back, in order, out of two pinned output slots.  Host and device memory
depend on the frame sizes and `chunk`, never on the length of the clip.  A chunk also ends where the source size changes
(every frame is CenterPad-ed to `size` on its own, so a folder may mix sizes); the clip continues across it.
"""
import queue
import threading
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import torch


def set_exemplar_rgb8(ctx, exemplar_rgb8, size):
    """test.py:57-66: CenterPad + CenterCrop to `size`, Lab, half size -> ctx.set_exemplar."""
    ref = torch.as_tensor(np.ascontiguousarray(exemplar_rgb8)).to(ctx.device)
    ctx.set_exemplar(ctx.resize_half(ctx.rgb8_to_lab(ctx.centerpad_rgb8(ref, size)[None])))


def _as_uint8_frame(x):
    a = np.ascontiguousarray(x.numpy() if isinstance(x, torch.Tensor) else x)
    if a.dtype != np.uint8 or a.ndim != 3 or a.shape[2] != 3:
        raise ValueError(f"a decoded frame must be uint8 [H,W,3], got {a.dtype} {a.shape}")
    return a


def colorize_stream(ctx, frames_iter, exemplar_rgb8, size, temperature=1e-10, wls=True, lam=500.0, sigma_color=4.0,
                    decode=None, chunk=16, workers=4, pin_memory=None):
    """Generator of colourised uint8 [size[0], size[1], 3] numpy frames, one per item of `frames_iter`, in order.

    Items are passed through `decode` (default: taken as they are) on `workers` threads; a decoded frame is a uint8
    [H,W,3] array or tensor.  An exception raised while decoding or on the device is raised here.  The exemplar
    (uint8 [H,W,3]) is installed with set_exemplar_rgb8 before the first frame."""
    if chunk < 1 or workers < 1:
        raise ValueError("chunk and workers must be >= 1")
    if pin_memory is None:
        pin_memory = torch.device(ctx.device).type == "cuda"
    decode = decode or (lambda item: item)
    set_exemplar_rgb8(ctx, exemplar_rgb8, size)

    done = object()
    results = queue.Queue(maxsize=1)     # (output slot, frame count) or an exception, to the caller
    free_out = threading.Semaphore(2)    # output slots the caller has finished reading
    stop = threading.Event()
    in_slots, out_slots = {}, {}

    def slot(slots, key, frame_shape, k):
        """The first k frames of slot `key`, (re)allocated for `chunk` frames of this shape."""
        t = slots.get(key)
        if t is None or tuple(t.shape[1:]) != frame_shape:
            t = torch.empty((chunk,) + frame_shape, dtype=torch.uint8)
            slots[key] = t = t.pin_memory() if pin_memory else t
        return t[:k]

    def put(item):
        while not stop.is_set():
            try:
                results.put(item, timeout=0.1)
                return True
            except queue.Full:
                pass
        return False

    def device_loop(pool):
        """Decodes run up to two chunks ahead; this thread gathers them in order and feeds the device."""
        try:
            pending, it = [], iter(frames_iter)
            exhausted, n_chunks, continue_clip = False, 0, False
            while True:
                while not exhausted and len(pending) < 2 * chunk:
                    try:
                        pending.append(pool.submit(lambda item: _as_uint8_frame(decode(item)), next(it)))
                    except StopIteration:
                        exhausted = True
                if not pending:
                    break
                first = pending[0].result()
                k, shape = 1, first.shape
                while k < min(chunk, len(pending)) and pending[k].result().shape == shape:
                    k += 1
                src = slot(in_slots, n_chunks & 1, shape, k)
                for i in range(k):
                    src[i].numpy()[...] = pending[i].result()
                del pending[:k]
                while not free_out.acquire(timeout=0.1):
                    if stop.is_set():
                        return
                out = slot(out_slots, n_chunks & 1, (size[0], size[1], 3), k)
                ctx.colorize_video_rgb8(src, size, temperature, wls, lam, sigma_color, continue_clip=continue_clip, out=out)
                continue_clip = True
                if not put((n_chunks & 1, k)):
                    return
                n_chunks += 1
            put(done)
        except BaseException as e:  # handed to the caller
            put(e)

    pool = ThreadPoolExecutor(max_workers=workers)
    worker = threading.Thread(target=device_loop, args=(pool,), daemon=True)
    worker.start()
    try:
        while True:
            item = results.get()
            if item is done:
                break
            if isinstance(item, BaseException):
                raise item
            s, k = item
            for i in range(k):
                yield out_slots[s][i].numpy().copy()
            free_out.release()
    finally:
        stop.set()
        worker.join()
        pool.shutdown(wait=True, cancel_futures=True)
