"""Throughput of the streaming path (dvc_colorize_video_rgb8) against the network pipeline alone (dvc_colorize_clip).

Seeded 1080 x 1920 uint8 frames, --image-size 960 1728: CenterPad takes its crop branch and the networks run at
480 x 864 (bench.py's size).  Seeded weights.  Every rate is taken over >= --seconds of wall time after a warm-up, with
the card's name and power limit read in the same run:

  (a) colorize_clip frames/s, pinned fp32 L in / ab out (the L of the same frames)
  (b) colorize_video_rgb8 frames/s, pinned uint8 in / out, WLS on and off; WLS on also for each post-processing batch G
  (c) device time per frame of dvc_postprocess_rgb8 over G frames vs the per-frame chain upsample2 -> l_to_guide8 ->
      fgs_filter -> lab_to_rgb8 (CUDA events)
  (d) tools/colorize_folder.py from a folder of PNGs to a folder of PNGs (wall time of the process, start-up included)

    python tools/stream_bench.py --out profiles/stream_bench.json
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "deep-exemplar-based-video-colorization_b200"))

import torch  # noqa: E402

HS, WS, SIZE = 1080, 1920, (960, 1728)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[torch.cuda.current_device()] if q.returncode == 0 else "unknown"


def seeded_frames(n, seed=0):
    g = torch.Generator().manual_seed(seed)
    base = torch.randint(0, 256, (n, HS // 8, WS // 8, 3), generator=g, dtype=torch.uint8)
    img = base.repeat_interleave(8, 1).repeat_interleave(8, 2).int()
    return (img + torch.randint(-6, 7, img.shape, generator=g)).clamp(0, 255).to(torch.uint8)


def rate(step, frames_per_step, seconds):
    """frames/s of `step` (which ends in a device synchronise) over >= `seconds`, after one warm-up step."""
    step()
    n, t0 = 0, time.perf_counter()
    while True:
        step()
        n += frames_per_step
        dt = time.perf_counter() - t0
        if dt >= seconds:
            return n / dt, n, dt


def device_ms(fn, reps):
    fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=2.0)
    ap.add_argument("--frames", type=int, default=32, help="distinct frames cycled through (one chunk = all of them)")
    ap.add_argument("--batches", type=int, nargs="*", default=[1, 2, 4, 8, 16], help="post-processing batch sizes G to sweep")
    ap.add_argument("--batch", type=int, default=8, help="the G the library ships with (dvc_ctx::video_batch)")
    ap.add_argument("--tool-frames", type=int, default=48)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("stream_bench needs a CUDA device")

    import dvc
    from dvc.stream import set_exemplar_rgb8
    from dvc.synth import make_state_dict

    ctx = dvc.get_context(0)
    for net, key in ((dvc.NET_VGG, "vgg"), (dvc.NET_WARP, "warp"), (dvc.NET_COLOR, "color")):
        ctx.set_weights(net, make_state_dict(key, seed=0))
    K = args.frames
    frames = seeded_frames(K).pin_memory()
    exemplar = seeded_frames(1, seed=1)[0]
    set_exemplar_rgb8(ctx, exemplar.numpy(), SIZE)
    res = {"card": card(), "source": [HS, WS], "image_size": list(SIZE), "nets": [SIZE[0] // 2, SIZE[1] // 2],
           "frames_per_call": K, "seconds_min": args.seconds, "host_cores": os.cpu_count()}

    # (a) the network pipeline alone, on the L of the same frames
    l, lh = ctx.ingest_rgb8(frames[:K].cuda(), SIZE)
    L = lh.cpu().pin_memory()
    ab = torch.empty(K, 2, SIZE[0] // 2, SIZE[1] // 2, dtype=torch.float32).pin_memory()
    fps, n, dt = rate(lambda: ctx.colorize_clip(L, 1e-10, out=ab), K, args.seconds)
    res["a_colorize_clip_fps"] = {"fps": fps, "frames": n, "s": dt}

    # (b) uint8 in, uint8 out
    out = torch.empty(K, SIZE[0], SIZE[1], 3, dtype=torch.uint8).pin_memory()

    def video(wls):
        return lambda: ctx.colorize_video_rgb8(frames, SIZE, wls=wls, continue_clip=True, out=out)

    ctx.colorize_video_rgb8(frames, SIZE, out=out)
    sweep = {}
    for G in args.batches:
        ctx.debug_flag("video_batch", G)
        fps, n, dt = rate(video(True), K, args.seconds)
        sweep[G] = {"fps": fps, "frames": n, "s": dt}
    res["b_video_wls_on_by_G"] = sweep
    G = args.batch
    ctx.debug_flag("video_batch", G)  # as shipped (DESIGN.md §4.5)
    for wls in (True, False):
        fps, n, dt = rate(video(wls), K, args.seconds)
        res[f"b_video_wls_{'on' if wls else 'off'}_fps"] = {"fps": fps, "frames": n, "s": dt}
    res["b_over_a_wls_on"] = res["b_video_wls_on_fps"]["fps"] / res["a_colorize_clip_fps"]["fps"]

    # (c) post-processing device time per frame: batched vs the per-frame chain
    abh = ab[:K].cuda()
    batched = device_ms(lambda: ctx.postprocess_rgb8(l[:G], abh[:G]), 20) / G

    def chain():
        up = ctx.upsample2_scaled(abh[:1], 1.25)
        up[0] = ctx.fgs_filter(ctx.l_to_guide8(l[0, 0]), up[0], 500.0, 4.0)
        ctx.lab_to_rgb8(l[:1], up)

    per_frame = device_ms(chain, 20)
    res["c_postprocess_ms_per_frame"] = {"batched_G": G, "batched": batched, "per_frame_chain": per_frame,
                                         "note": "the per-frame chain includes the host sync of each dvc_fgs_filter call"}

    # (d) the whole tool, PNG folder -> PNG folder
    from PIL import Image

    with tempfile.TemporaryDirectory() as tmp:
        src, dst = os.path.join(tmp, "in"), os.path.join(tmp, "out")
        os.makedirs(src)
        fr = seeded_frames(args.tool_frames, seed=2).numpy()
        for i, f in enumerate(fr):
            Image.fromarray(f).save(os.path.join(src, f"{i:05d}.png"), compress_level=1)
        Image.fromarray(exemplar.numpy()).save(os.path.join(tmp, "ref.png"))
        workers = min(8, os.cpu_count() or 1)
        t0 = time.perf_counter()
        subprocess.run([sys.executable, os.path.join(ROOT, "tools", "colorize_folder.py"), "--clip", src, "--ref",
                        os.path.join(tmp, "ref.png"), "--out", dst, "--seeded-weights", "--image-size", str(SIZE[0]), str(SIZE[1]),
                        "--workers", str(workers)], check=True)
        dt = time.perf_counter() - t0
        res["d_tool"] = {"frames": args.tool_frames, "s": dt, "fps": args.tool_frames / dt, "workers": workers,
                         "host_cores": os.cpu_count(), "note": "process wall time, CUDA and model start-up included"}

    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
