"""Generate tests/golden/*.npz from the UNMODIFIED reference (run in the build container only).

    python oracle/make_golden.py            # writes tests/golden/, prints the pin report

For every case the real reference modules (imported read-only from /root/reference through
oracle/ref_import.py) run `frame_colorization` on seeded weights (oracle/weights.py) and seeded
inputs in fp32 (the reference's own arithmetic) and in fp64 (same modules, .double()).  The
restatement in oracle/dvc_oracle.py is run on the same tensors and must agree BIT-EXACTLY with
the fp32 reference (same torch ops in the same order) -- that is the pin.  What is stored:
inputs, the fp32 reference outputs, the fp64 outputs and the fp64 top-2 correlation gap per query
row (for the tie-aware metric of SURVEY.md §8c).

Cases (all legal shapes: H % 8 == 0, W % 16 == 0):
  small_32x48      B=1, T=1e-10            every intermediate stored
  padbranch_40x64  B=1, T=1e-10            H % 16 == 8 -> NonlocalNet.py:461-463 replicate-pad branch
  softmax_32x64    B=1, T=0.01             FrameColor.py:52 default temperature (true softmax)
  softmax5_48x48   B=1, T=0.005            NonlocalNet.py:438 default temperature
  batch2_32x32     B=2, T=1e-10            batched call (squeeze_/broadcast behaviour, NonlocalNet.py:488,496)
  clip3_32x48      3-frame recurrence      test.py:76-96 semantics (I_last feeds the next frame)
  default_216x384  B=1, T=1e-10            test.py's default processing resolution; outputs only
  cfg1_256x256     B=1, T=1e-10            BASELINE.json configs[0]; outputs only, inputs regenerated from the seed
  default_480x864  B=1, T=1e-10            BASELINE.json configs[1], the bench size (N = 25920); outputs only, inputs
                                           regenerated from the seed (make_lab(seed), make_lab(seed+1), make_lab(seed+2)*0.5)
  contextual_loss  ContextualLoss_forward  models/ContextualLoss.py on the seeded maps of contextual_loss_maps(); outputs only

    python oracle/make_golden.py --only default_480x864     # (re)generate one case, keep the others untouched
"""
import os
import sys
import time

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

from oracle import dvc_oracle as O  # noqa: E402
from oracle import ref_import  # noqa: E402
from oracle.weights import make_lab, make_state_dict  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
KEYS = ["r12", "r22", "r32", "r42", "r52"]


def ref_frame(ns, mods, IA, IB, last, T):
    vgg, warp, color = mods
    with torch.no_grad():
        rgb = ns.tensor_lab2rgb(torch.cat((ns.uncenter_l(IB[:, 0:1]), IB[:, 1:3]), dim=1))
        fB = vgg(rgb, KEYS, preprocess=True)
        ab, warped, fA = ns.frame_colorization(IA, IB, last, fB, vgg, warp, color, feature_noise=0, temperature=T)
        # similarity map is not returned by frame_colorization; recompute it through the module itself
        An = [ns.feature_normalize(t) for t in fA[1:]]
        Bn = [ns.feature_normalize(t) for t in fB[1:]]
        _, sim = warp(IB, *An, *Bn, temperature=T)
    return dict(ab=ab, warped=warped, sim=sim, fA=fA, fB=fB)


def oracle_frame(sds, IA, IB, last, T):
    ex = {}
    with torch.no_grad():
        fB = O.exemplar_features(sds["vgg"], IB)
        ab, warped, sim, fA = O.frame_colorization(sds, IA, IB, last, fB, temperature=T, extras=ex)
    return dict(ab=ab, warped=warped, sim=sim, fA=fA, fB=fB, **ex)


def npf(t):
    return t.detach().cpu().numpy()


def run_case(ns, name, B, H, W, T, seed, store_all, store_inputs=True):
    torch.set_num_threads(8)
    sds32 = {k: make_state_dict(k, seed=0) for k in ("vgg", "warp", "color")}
    sds64 = {k: O._cast(v, torch.float64) for k, v in sds32.items()}
    IA = make_lab(seed, B, H, W)
    IB = make_lab(seed + 1, B, H, W)
    last = make_lab(seed + 2, B, H, W) * 0.5
    mods32 = ref_import.build_modules(ns, sds32)
    mods64 = ref_import.build_modules(ns, sds32, torch.float64)
    r32 = ref_frame(ns, mods32, IA, IB, last, T)
    r64 = ref_frame(ns, mods64, IA.double(), IB.double(), last.double(), T)
    o32 = oracle_frame(sds32, IA, IB, last, T)
    o64 = oracle_frame(sds64, IA.double(), IB.double(), last.double(), T)
    report = {}
    for k in ("ab", "warped", "sim"):
        report[f"oracle32_vs_ref32_{k}"] = float((o32[k] - r32[k]).abs().max())
        report[f"oracle64_vs_ref64_{k}"] = float((o64[k] - r64[k]).abs().max())
        report[f"ref32_vs_ref64_{k}"] = float((r32[k].double() - r64[k]).abs().max())
    for i, k in enumerate(KEYS):
        report[f"oracle32_vs_ref32_{k}"] = float((o32["fA"][i] - r32["fA"][i]).abs().max())
        report[f"oracle32_vs_ref32_B_{k}"] = float((o32["fB"][i] - r32["fB"][i]).abs().max())
    gap = O.top2_gap(o64["theta_hat"], o64["phi_hat"])
    report["rows_gap_lt_1e-6"] = int((gap < 1e-6).sum())
    report["argmax_mismatch_32_vs_64"] = int((o32["argmax"] != o64["argmax"]).sum())
    out = dict(
        temperature=np.float64(T), seed=np.int64(seed),
        ab32=npf(r32["ab"]), warped32=npf(r32["warped"][:, :, ::4, ::4]), sim32=npf(r32["sim"][:, :, ::4, ::4]),
        ab64=npf(r64["ab"]), warped64=npf(r64["warped"][:, :, ::4, ::4]), sim64=npf(r64["sim"][:, :, ::4, ::4]),
        argmax64=npf(o64["argmax"]).astype(np.int32), gap64=npf(gap).astype(np.float32),
    )
    if store_inputs:
        out.update(IA_lab=npf(IA), IB_lab=npf(IB), IA_last_lab=npf(last))
    else:
        # Teacher-forced fp32 ColorVidNet on the fp64 warp / similarity (FrameColor.py:63-65): at these sizes a single
        # near-tie row whose fp32 and fp64 argmax differ changes the warped colour and, through ColorVidNet, ab32 by
        # O(10); the noise floor of the colour network itself is |ab32_tf - ab64|.
        up = lambda t: torch.nn.functional.interpolate(t, scale_factor=4, mode="nearest")
        with torch.no_grad():
            x_tf = torch.cat((IA[:, 0:1], r64["warped"][:, 1:3].float(), r64["sim"].float(), last), 1)
            ab32_tf = mods32[2](x_tf)
            o_tf = O.colorvidnet_forward(sds32["color"], x_tf)
        report["oracle32_vs_ref32_ab_tf"] = float((o_tf - ab32_tf).abs().max())
        report["ref32tf_vs_ref64_ab"] = float((ab32_tf.double() - r64["ab"]).abs().max())
        out["ab32_tf"] = npf(ab32_tf)
        out["argmax32"] = npf(o32["argmax"]).astype(np.int32)
    if store_all:
        for i, k in enumerate(KEYS):
            out[f"A_{k}"] = npf(r32["fA"][i])
            out[f"B_{k}"] = npf(r32["fB"][i])
        out["theta_hat32"] = npf(o32["theta_hat"])
        out["phi_hat32"] = npf(o32["phi_hat"])
        out["theta_hat64"] = npf(o64["theta_hat"]).astype(np.float64)
        out["phi_hat64"] = npf(o64["phi_hat"]).astype(np.float64)
        out["V32"] = npf(o32["V"])
    np.savez_compressed(os.path.join(GOLD, name + ".npz"), **out)
    return report


def run_clip(ns, name, F_, H, W, seed):
    sds32 = {k: make_state_dict(k, seed=0) for k in ("vgg", "warp", "color")}
    frames = torch.cat([make_lab(seed + 10 * t, 1, H, W) for t in range(F_)], 0)
    IB = make_lab(seed + 1, 1, H, W)
    mods = ref_import.build_modules(ns, sds32)
    vgg, warp, color = mods
    outs = []
    with torch.no_grad():
        rgb = ns.tensor_lab2rgb(torch.cat((ns.uncenter_l(IB[:, 0:1]), IB[:, 1:3]), dim=1))
        fB = vgg(rgb, KEYS, preprocess=True)
        last = torch.zeros_like(frames[0:1])
        for t in range(F_):
            IA = frames[t:t + 1]
            ab, _, _ = ns.frame_colorization(IA, IB, last, fB, vgg, warp, color, feature_noise=0, temperature=1e-10)
            last = torch.cat((IA[:, 0:1], ab), dim=1)
            outs.append(ab)
        ref = torch.cat(outs, 0)
        mine = O.colorize_clip(sds32, frames, IB)
    np.savez_compressed(os.path.join(GOLD, name + ".npz"), frames_lab=npf(frames), IB_lab=npf(IB), ab32=npf(ref))
    return {"oracle32_vs_ref32_ab": float((mine - ref).abs().max())}


def contextual_loss_maps():
    """(key, X, Y, feature_centering) of the contextual-loss case: seeded ReLU feature maps of several depths."""
    g = torch.Generator().manual_seed(31)
    for (B, C, h, w) in ((2, 128, 12, 16), (1, 256, 16, 16), (1, 512, 8, 12)):
        X = torch.relu(torch.randn(B, C, h, w, generator=g))
        Y = torch.relu(torch.randn(B, C, h, w, generator=g) + 0.3 * X)
        for centering in (True, False):
            yield f"loss_{C}_{int(centering)}", X, Y, centering


def run_contextual_loss(ns, name):
    torch.set_num_threads(8)
    mod = ns.ContextualLoss_forward()
    out, report = {}, {}
    with torch.no_grad():
        for key, X, Y, centering in contextual_loss_maps():
            ref = mod(X.clone(), Y.clone(), 0.1, centering)
            report[f"oracle32_vs_ref32_{key}"] = float((O.contextual_loss_forward(X, Y, 0.1, centering) - ref).abs().max())
            out[key] = npf(ref)
    np.savez_compressed(os.path.join(GOLD, name + ".npz"), **out)
    return report


def write_report(lines, replace_all):
    """PIN_REPORT.txt: one section per case; --only replaces just that case's section."""
    path = os.path.join(GOLD, "PIN_REPORT.txt")
    head = "Pin report written by oracle/make_golden.py (torch %s, %d threads)\n" % (torch.__version__, torch.get_num_threads())
    sections = {}
    order = []
    if not replace_all and os.path.isfile(path):
        cur = None
        for ln in open(path).read().splitlines()[1:]:
            if ln.startswith("["):
                cur = ln.strip()[1:-1]
                sections[cur] = []
                order.append(cur)
            elif cur is not None:
                sections[cur].append(ln)
    for name, rep in lines:
        if name not in sections:
            order.append(name)
        sections[name] = [f"    {k:36s} {v}" for k, v in rep.items()]
    with open(path, "w") as f:
        f.write(head)
        for name in order:
            f.write(f"[{name}]\n")
            for ln in sections[name]:
                f.write(ln + "\n")


def main():
    import argparse

    ap = argparse.ArgumentParser()
    ap.add_argument("--only", default=None, help="generate just this case (the other files stay untouched)")
    args = ap.parse_args()
    os.makedirs(GOLD, exist_ok=True)
    ns = ref_import.load()
    cases = [
        ("small_32x48", 1, 32, 48, 1e-10, 101, True),
        ("padbranch_40x64", 1, 40, 64, 1e-10, 202, True),
        ("softmax_32x64", 1, 32, 64, 0.01, 303, False),
        ("softmax5_48x48", 1, 48, 48, 0.005, 404, False),
        ("batch2_32x32", 2, 32, 32, 1e-10, 505, False),
        ("default_216x384", 1, 216, 384, 1e-10, 606, False),
        ("cfg1_256x256", 1, 256, 256, 1e-10, 808, False),
        ("default_480x864", 1, 480, 864, 1e-10, 909, False),
    ]
    big = {"cfg1_256x256", "default_480x864"}  # inputs are regenerated from the seed by the tests
    lines = []
    for name, B, H, W, T, seed, store_all in cases:
        if args.only and name != args.only:
            continue
        t0 = time.time()
        rep = run_case(ns, name, B, H, W, T, seed, store_all, store_inputs=name not in big)
        lines.append((name, rep))
        print(f"[{name}] {time.time() - t0:.1f}s")
        for k, v in rep.items():
            print(f"    {k:36s} {v}")
    if not args.only or args.only == "clip3_32x48":
        rep = run_clip(ns, "clip3_32x48", 3, 32, 48, 707)
        print("[clip3_32x48]", rep)
        lines.append(("clip3_32x48", rep))
    if not args.only or args.only == "contextual_loss":
        rep = run_contextual_loss(ns, "contextual_loss")
        print("[contextual_loss]", rep)
        lines.append(("contextual_loss", rep))
    write_report(lines, replace_all=not args.only)


if __name__ == "__main__":
    main()
