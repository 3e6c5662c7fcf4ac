"""The reference's test.py:29-125 data flow on the device, using only libdvc entry points (no reference code):

    PNG files decoded on a thread pool -> chunks of uint8 frames (dvc/stream.py: colorize_stream) -> per chunk one
    dvc_colorize_video_rgb8 call: CenterPad + CenterCrop to --image_size, Lab, 1/2 resolution (dvc_ingest_rgb8) -> per
    frame VGG19 / WarpNet / correlation / ColorVidNet with the recurrence kept on the device (the dvc_colorize_clip
    driver) -> ab x2 * 1.25 -> WLS filter guided by the full-resolution luminance (test.py:105-112) -> sRGB uint8
    (dvc_postprocess_rgb8) -> PNG files.  The exemplar goes through dvc_resize_antialias_crop_rgb8 -> dvc_rgb8_to_lab ->
    dvc_resize_half -> dvc_set_exemplar once.  Memory does not grow with the length of the clip.

    python tools/colorize_folder.py --clip frames/ --ref exemplar.png --out out/ \
        --vgg vgg19_conv.pth --warp nonlocal_net_iter_76000.pth --color colornet_iter_76000.pth

What the reference does and this script does not: the AVI writer (folder2vid).  Image decode / encode stays on the host
(PIL), as in the reference.  Without checkpoints (none ship with the reference tree) pass --seeded-weights to run the
pipeline on the seeded random weights of dvc/synth.py (useful as a smoke run only).
"""
import argparse
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "deep-exemplar-based-video-colorization_b200"))

import numpy as np
import torch


def load_rgb8(path):
    from PIL import Image

    return torch.from_numpy(np.asarray(Image.open(path).convert("RGB"), dtype=np.uint8).copy())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--clip", required=True, help="folder of frames (sorted by the digits in the file names, test.py:41)")
    ap.add_argument("--ref", required=True, help="exemplar image (same size as the frames)")
    ap.add_argument("--out", required=True)
    ap.add_argument("--vgg"), ap.add_argument("--warp"), ap.add_argument("--color")
    ap.add_argument("--seeded-weights", action="store_true")
    ap.add_argument("--temperature", type=float, default=1e-10)  # test.py:94
    ap.add_argument("--image-size", type=int, nargs=2, default=[216 * 2, 384 * 2], help="test.py:132")
    ap.add_argument("--no-wls", action="store_true", help="skip the Fast Global Smoother (test.py:31 wls_filter_on)")
    ap.add_argument("--lambda-value", type=float, default=500.0)  # test.py:32
    ap.add_argument("--sigma-color", type=float, default=4.0)    # test.py:33
    ap.add_argument("--workers", type=int, default=min(8, os.cpu_count() or 1), help="PNG decode threads")
    args = ap.parse_args()

    import dvc
    from dvc.synth import make_state_dict

    ctx = dvc.get_context(0)
    for net, key, path in ((dvc.NET_VGG, "vgg", args.vgg), (dvc.NET_WARP, "warp", args.warp), (dvc.NET_COLOR, "color", args.color)):
        if path:
            ctx.set_weights(net, torch.load(path, map_location="cpu"))
        elif args.seeded_weights:
            ctx.set_weights(net, make_state_dict(key, seed=0))
        else:
            raise SystemExit(f"--{key} checkpoint missing (or pass --seeded-weights)")

    names = sorted(os.listdir(args.clip), key=lambda f: int("".join(filter(str.isdigit, f)) or -1))
    H, W = args.image_size
    if H % 16 or W % 32:
        raise SystemExit("--image-size must have H % 16 == 0 and W % 32 == 0 (the networks run at half of it)")
    from PIL import Image

    from dvc.stream import colorize_stream

    os.makedirs(args.out, exist_ok=True)
    frames = colorize_stream(ctx, (os.path.join(args.clip, n) for n in names), load_rgb8(args.ref), (H, W), args.temperature,
                             wls=not args.no_wls, lam=args.lambda_value, sigma_color=args.sigma_color, decode=load_rgb8,
                             workers=args.workers)
    for n, img in zip(names, frames):
        Image.fromarray(img).save(os.path.join(args.out, os.path.splitext(n)[0] + ".png"))
    print(f"{len(names)} frames -> {args.out}")


if __name__ == "__main__":
    main()
