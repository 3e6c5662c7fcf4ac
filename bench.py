#!/usr/bin/env python
"""480p frames/sec of the exemplar-colorization forward path on N B200s + correlation-kernel roofline.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): one 480x854 grayscale frame + 1 exemplar, replicate-padded to the
legal 480x864 (SURVEY.md fact 2: the reference rejects W % 16 != 0), N = 120*216 = 25920 positions.
A "step" = one frame through the whole hot path (VGG19 -> WarpNet -> correlation/softmax/warp -> ColorVidNet,
FrameColor.py:41-67) with the frame-to-frame recurrence of test.py:96.  Under torchrun each rank owns its own
contiguous segment of frames (weak scaling: K frames per rank) and rank 0's exemplar operands are broadcast
once over NCCL before the timed region (SURVEY.md §8e).

Timed legs (own arm):
  value : frames already resident in HBM, dvc_colorize_clip on device buffers, CUDA events.
  e2e   : the public clip API (dvc_colorize_clip) on PINNED HOST buffers: every step copies one L frame
          host->device and the predicted ab device->host inside the timed region.
  roofline : every tensor-core convolution launch (the dominant kernel, ~78 % of the device time) and, as roofline_corr, the
          correlation (K7), timed with CUDA events on the launching stream in a single-stream pass inside this run;
          achieved = algorithmic FLOPs / launch time against the measured dense-bf16 peak (burst: the pass lasts ~35 ms).
  sustained : the `value` leg back to back for >= 2.5 s with its own clock samples.
  clip64 : BASELINE configs[2], 64 frames in N segments, exemplar prologue + NCCL broadcast inside the wall clock.
  rank_checksum : every rank colourises one common frame; the bit patterns must agree across ranks or the run aborts.
  cpu_baseline : the CPU oracle (port of the reference's PyTorch forward) on the host cores, bounded sample.
Reference arm (--impl reference): the same CPU oracle timed step by step on rank 0 (the reference is pure
Python/PyTorch and cannot travel to the GPU box; oracle/dvc_oracle.py is bit-exact with it, tests/golden/PIN_REPORT.txt).

--dump-outputs DIR: after the timed steps, rank 0 writes what the timed path returned for its last step, DIR/ab.npy
(float32 [1,2,480,864], 3.3 MB).  Inputs and weights are seeded, so two builds run with the same arguments can be
compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "deep-exemplar-based-video-colorization_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

H, W_RAW, W = 480, 854, 864
N_POS = (H // 4) * (W // 4)
CORR_FLOP = 2.0 * N_POS * N_POS * (256 + 3)  # SURVEY.md §8d
TEMPERATURE = 1e-10  # test.py:94
METRIC = "480p frames/sec"
# the same string in both arms (own and --impl reference): both run the recurrence of test.py:96 over a contiguous segment
WORKLOAD = ("480x854 frame padded to 480x864 + 1 exemplar, full forward path (FrameColor.py:41-67), T=1e-10, "
            "batch 1 with the frame recurrence of test.py:96; one contiguous K-frame segment per process")


def synth_frames(n, seed0):
    """L-channel frames [n,1,480,864]: 480x854 synthetic content, replicate-padded on the right to 864."""
    from dvc.synth import make_lab

    out = []
    for t in range(n):
        lab = make_lab(seed0 + t, 1, H, W_RAW)
        out.append(torch.nn.functional.pad(lab[:, 0:1], (0, W - W_RAW, 0, 0), mode="replicate"))
    return torch.cat(out, 0)


def synth_exemplar(seed=4321):
    from dvc.synth import make_lab

    return torch.nn.functional.pad(make_lab(seed, 1, H, W_RAW), (0, W - W_RAW, 0, 0), mode="replicate")


class ClockSampler:
    """nvidia-smi clocks / power / throttle reasons streamed DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self._t = threading.Thread(target=self._pump, daemon=True)
            self._t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def stop(self, windows=None):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        time.sleep(0.06)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=3)
        except Exception:
            self.proc.kill()
        inside = lambda t: windows is None or any(b <= t <= e + 0.06 for b, e in windows)
        rows = [l.split(",") for t, l in self.lines if inside(t)]
        rows = [[x.strip() for x in r] for r in rows if len(r) >= 7]
        sm = sorted(int(r[0]) for r in rows if r[0].isdigit())
        mx = [int(r[1]) for r in rows if r[1].isdigit()]
        pw = [float(r[2]) for r in rows if r[2].replace(".", "", 1).isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in rows for n, v in zip(names, r[3:7]) if v.lower() == "active"})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_min_mhz": sm[0] if sm else None,
                "sm_max_mhz": max(mx) if mx else None, "power_w_max": max(pw) if pw else None, "reasons": reasons,
                "samples": len(rows)}


def ncu_traffic(kernel):
    """DRAM bytes of one launch from the committed ncu --set full capture (profiles/), or None."""
    path = os.path.join(ROOT, "profiles", "ncu_r2_traffic.json")
    try:
        return json.load(open(path))[kernel]["bytes"]
    except Exception:
        return None


def measured_peak(window_s):
    """Dense bf16 peak to hold a kernel against: the BURST figure when the kernels were timed in a short window (the
    per-kernel leg lasts tens of milliseconds: the chip has not reached its power-limited steady state), the SUSTAINED
    one for a window of a second or more (MEASURED_PEAKS.json; B200_PROFILING.md fallback otherwise)."""
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    burst = window_s < 1.0
    if os.path.isfile(path):
        d = json.load(open(path))
        if burst and "bf16_tflops" in d:
            return float(d["bf16_tflops"]), f"measured bf16 dense, burst (MEASURED_PEAKS.json; timed window {window_s * 1e3:.0f} ms)"
        return (float(d.get("bf16_tflops_sustained", d.get("bf16_tflops"))),
                f"measured bf16 dense, sustained (MEASURED_PEAKS.json; timed window {window_s:.1f} s)")
    return (1700.0, "fallback burst (B200_PROFILING.md)") if burst else (1400.0, "fallback (B200_PROFILING.md: ~1.4 PFLOP/s sustained)")


def pick_cpu_threads(sds):
    """torch's CPU kernels stop scaling (and regress) well before 128 SMT threads on this workload: try a few
    intra-op thread counts on a quarter-size ColorVidNet forward and keep the fastest (a few seconds)."""
    from oracle import dvc_oracle as O

    cores = os.cpu_count() or 1
    cands = sorted({c for c in (8, 16, 32, 64, cores) if c <= cores})
    x = torch.randn(1, 7, H // 2, W // 2)
    best, best_t = cands[0], float("inf")
    with torch.no_grad():
        for c in cands:
            torch.set_num_threads(c)
            O.colorvidnet_forward(sds["color"], x)
            t0 = time.perf_counter()
            O.colorvidnet_forward(sds["color"], x)
            dt = time.perf_counter() - t0
            if dt < best_t:
                best, best_t = c, dt
    torch.set_num_threads(best)
    return best


def dump_outputs(out_dir, **arrays):
    """--dump-outputs: every array as out_dir/<name>.npy in float32."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().to(torch.float32).cpu().numpy())


def cpu_frames_per_sec(n_timed, warm=1):
    """The CPU oracle (= the reference's PyTorch CPU forward, bit-exact port) on this host's cores.
    Returns the step times, the thread count and the ab of the last step."""
    from dvc.synth import make_state_dict
    from oracle import dvc_oracle as O

    sds = {k: make_state_dict(k, seed=0) for k in ("vgg", "warp", "color")}
    cores = pick_cpu_threads(sds)
    IB = synth_exemplar()
    frames = synth_frames(warm + n_timed, 1000)
    times = []
    with torch.no_grad():
        fB = O.exemplar_features(sds["vgg"], IB)
        last = torch.zeros(1, 3, H, W)
        for t in range(warm + n_timed):
            IA = torch.cat((frames[t:t + 1], torch.zeros(1, 2, H, W)), 1)
            t0 = time.perf_counter()
            ab, _, _, _ = O.frame_colorization(sds, IA, IB, last, fB, temperature=TEMPERATURE, row_chunk=4096)
            dt = time.perf_counter() - t0
            if t >= warm:
                times.append(dt)
            last = torch.cat((frames[t:t + 1], ab), 1)
    return times, cores, ab


def run_reference(args, rank):
    """--impl reference: the reference's CPU path (oracle port) timed step by step on rank 0."""
    if rank != 0:
        return
    t_all = time.perf_counter()
    times, cores, ab = cpu_frames_per_sec(args.steps, warm=max(args.warmup, 1))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, ab=ab)
    total = sum(times)
    fps = len(times) / total
    line = {
        "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * total / len(times), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "impl": "reference",
        "config": {"workload": WORKLOAD, "N_positions": N_POS, "weights": "seeded random (dvc/synth.py), no checkpoint available",
                   "note": "the reference arm is ONE CPU process on rank 0's host cores whatever --gpus says (the reference "
                           "has no multi-GPU inference path, SURVEY.md §8e): at N > 1 the driver's ratio is N GPUs vs one host run"},
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores, "kind": "port",
                         "sample": f"{len(times)} frames of the workload, one per step, torch {torch.__version__} CPU"},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "wall_s": time.perf_counter() - t_all,
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="own", choices=["own", "reference"])
    ap.add_argument("--corr-math", default=os.environ.get("DVC_CORR_MATH", "fp16x3"), choices=["fp32", "tf32x3", "bf16x3", "fp16x3"])
    ap.add_argument("--conv-math", default=os.environ.get("DVC_CONV_MATH", "tf32x3"), choices=["fp32", "tf32x3"])
    ap.add_argument("--tc-kc", type=int, default=int(os.environ.get("DVC_TC_KC", "1")),
                    help="k-blocks summed in TMEM before promotion to fp32 registers (1 = parity mode)")
    ap.add_argument("--tc-kbytes", type=int, default=int(os.environ.get("DVC_TC_KBYTES", "128")), choices=[64, 128],
                    help="K bytes per pipeline stage of the conv engine (64 = twice the stages, measured slower)")
    ap.add_argument("--tc-f16", type=int, default=int(os.environ.get("DVC_TC_F16", "1")),
                    help="1: convolutions with bounded inputs run 3xFP16 on scaled planes; 0: 3xTF32 everywhere")
    ap.add_argument("--corr-screen", type=int, default=int(os.environ.get("DVC_CORR_SCREEN", "1")), choices=[0, 1],
                    help="1 = T->0 correlation as one fp16 screening pass + exact fp32 re-scoring of the candidates; 0 = exact 3-pass kernel")
    ap.add_argument("--corr-cluster", type=int, default=int(os.environ.get("DVC_CORR_CLUSTER", "2")), choices=[1, 2],
                    help="2 = CTA pairs (tcgen05.mma.cta_group::2) in the correlation kernel, 1 = single CTAs")
    ap.add_argument("--tc-tail", type=int, default=int(os.environ.get("DVC_TC_TAIL", "0")),
                    help="1: partial last rounds of 256-channel conv launches run on 128-channel tiles; 0: off")
    ap.add_argument("--tc-splits", type=int, default=int(os.environ.get("DVC_TC_SPLITS", "1")),
                    help="split-K of the conv engine: 1 off (default), 0 automatic")
    ap.add_argument("--tc-rowshare", type=int, default=int(os.environ.get("DVC_TC_ROWSHARE", "0")), choices=[0, 1],
                    help="1: the taps of a 3x3 kernel row share one activation tile in shared memory (conv_tc.cu: CfgRS)")
    ap.add_argument("--clip-astreams", type=int, default=int(os.environ.get("DVC_CLIP_ASTREAMS", "1")), choices=[1, 2],
                    help="2: the frame-independent phase of frames t+1 and t+2 overlaps frame t's ColorVidNet (two streams)")
    ap.add_argument("--tc-cluster", type=int, default=int(os.environ.get("DVC_TC_CLUSTER", "2")), choices=[1, 2],
                    help="2 = CTA pairs (tcgen05.mma.cta_group::2) in the conv engine, 1 = single CTAs")
    ap.add_argument("--cpu-sample", type=int, default=4, help="frames timed for cpu_baseline (0 = skip)")
    ap.add_argument("--sustain-s", type=float, default=2.5, help="length of the extra sustained run of the headline (0 = skip)")
    ap.add_argument("--clip-frames", type=int, default=64, help="frames of the config-3 clip (0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "own" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch.distributed as dist

    import dvc
    from dvc.clip import prepare_exemplar
    from dvc.synth import make_state_dict

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: libdvc has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ctx = dvc.get_context(local)
    for net, key in ((dvc.NET_VGG, "vgg"), (dvc.NET_WARP, "warp"), (dvc.NET_COLOR, "color")):
        ctx.set_weights(net, make_state_dict(key, seed=0))
    corr_mode = {"fp32": dvc.MATH_FP32, "tf32x3": dvc.MATH_TF32X3, "bf16x3": dvc.MATH_BF16X3, "fp16x3": dvc.MATH_FP16X3}[args.corr_math]
    ctx.set_math(conv=dvc.MATH_TF32X3 if args.conv_math == "tf32x3" else dvc.MATH_FP32, corr=corr_mode)
    ctx.debug_flag("tc_kc", args.tc_kc)
    ctx.debug_flag("tc_cluster", args.tc_cluster)
    ctx.debug_flag("tc_kbytes", args.tc_kbytes)
    ctx.debug_flag("tc_splits", args.tc_splits)
    ctx.debug_flag("tc_f16", args.tc_f16)
    ctx.debug_flag("tc_tail", args.tc_tail)
    ctx.debug_flag("tc_rowshare", args.tc_rowshare)
    ctx.debug_flag("clip_astreams", args.clip_astreams)
    ctx.debug_flag("corr_cluster", args.corr_cluster)
    ctx.debug_flag("corr_screen", args.corr_screen)

    K, Wm = args.steps, args.warmup
    # every rank owns its own contiguous segment of synthetic frames (distinct content per rank and per step)
    host_L = synth_frames(Wm + K, 1000 + 10000 * rank).pin_memory()
    IB = synth_exemplar()
    t0 = time.perf_counter()
    prepare_exemplar(ctx, IB, H, W, src=0)  # rank 0: exemplar prologue; NCCL broadcast of the operand pack
    torch.cuda.synchronize()
    exemplar_ms = 1e3 * (time.perf_counter() - t0)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---------------- leg 1: inputs resident in HBM (same clip API, device buffers) ----------------
    dev_L = host_L.cuda()
    dev_out = torch.empty(K, 2, H, W, device="cuda")
    ctx.colorize_clip(dev_L[:Wm].contiguous(), TEMPERATURE)  # W warm-up frames
    barrier()
    ctx.launch_count(True)
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
        time.sleep(0.12)  # let the first samples arrive; they are filtered to the timed window below
    t_begin = time.perf_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    ctx.colorize_clip(dev_L[Wm:Wm + K], TEMPERATURE, out=dev_out)  # K frames, recurrence of test.py:96 on the device
    e1.record()
    barrier()
    t_end = time.perf_counter()
    ms_dev = max_over_ranks(e0.elapsed_time(e1))
    launches = ctx.launch_count(True)

    # ---------------- leg 2: end to end through the clip API with host buffers ----------------
    host_out = torch.empty(K, 2, H, W).pin_memory()
    ctx.colorize_clip(host_L[:Wm].contiguous().pin_memory(), TEMPERATURE)
    barrier()
    seg = host_L[Wm:Wm + K]
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_begin2 = time.perf_counter()
    e2.record()
    ctx.colorize_clip(seg, TEMPERATURE, out=host_out)  # per frame: H2D of L, full path, D2H of ab
    e3.record()
    barrier()
    t_end2 = time.perf_counter()
    ms_e2e = max_over_ranks(e2.elapsed_time(e3))
    # clocks / throttle reasons sampled inside the two timed regions (value leg and e2e leg)
    clocks = sampler.stop([(t_begin, t_end), (t_begin2, t_end2)]) if sampler else None

    # ---------------- multi-GPU correctness: every rank colourises ONE common frame with its (imported) exemplar pack ----
    # outside the timed regions; the ab bit patterns must agree across ranks (same kernels, same operands), else abort
    common_L = synth_frames(1, 777).cuda()
    ab_c = ctx.colorize_frames(common_L, torch.zeros(1, 3, H, W, device="cuda"), TEMPERATURE)
    bits = ab_c.view(torch.int32).to(torch.int64)
    check = torch.stack((bits.sum(), (bits * (torch.arange(bits.numel(), device="cuda").view_as(bits) % 8191 + 1)).sum()))
    checks = [check]
    if world > 1:
        checks = [torch.zeros_like(check) for _ in range(world)]
        dist.all_gather(checks, check)
    rank_check_ok = all(torch.equal(c_, checks[0]) for c_ in checks)
    if not rank_check_ok:
        raise SystemExit(f"rank {rank}: the common-frame checksum differs between ranks ({[c_.tolist() for c_ in checks]}): "
                         "a corrupt exemplar import or a non-deterministic kernel -- no number is printed")
    if not (torch.isfinite(ab_c).all() and float(ab_c.abs().max()) <= 128.0):
        raise SystemExit("common frame: ab out of range")

    # ---------------- config 3 (BASELINE.json configs[2]): a 64-frame clip, one contiguous segment per GPU, wall time
    # INCLUDING the exemplar prologue and its NCCL broadcast on the warm communicator (SURVEY.md §8d) ----------------
    clip64 = None
    if args.clip_frames > 0:
        from dvc.clip import segment_bounds

        F_clip = args.clip_frames
        s0, s1 = segment_bounds(F_clip, world, rank)
        clip_L = synth_frames(s1 - s0, 50000 + s0).pin_memory() if s1 > s0 else None
        clip_out = torch.empty(max(s1 - s0, 1), 2, H, W).pin_memory()
        barrier()
        t_c0 = time.perf_counter()
        prepare_exemplar(ctx, IB, H, W, src=0)
        if clip_L is not None:
            ctx.colorize_clip(clip_L, TEMPERATURE, out=clip_out[: s1 - s0])
        barrier()
        clip_ms = max_over_ranks(1e3 * (time.perf_counter() - t_c0))
        clip64 = {"frames": F_clip, "segments": world, "wall_ms": clip_ms, "frames_per_s": F_clip / (clip_ms * 1e-3),
                  "includes": "exemplar prologue (VGG19 + WarpNet B side) on rank 0, NCCL broadcast of the 27 MB operand "
                              "pack, per-frame H2D / D2H through dvc_colorize_clip; host wall clock between barriers, max over ranks"}

    # ---------------- sustained run of the headline leg (>= 2 s of back-to-back frames, clocks sampled) ----------------
    sustained = None
    if args.sustain_s > 0:
        n_s = max(K, int(args.sustain_s * K / (ms_dev * 1e-3)) + 1)
        n_s = min(n_s, 1200)
        reps = (n_s + K - 1) // K
        long_L = dev_L[Wm:Wm + K].repeat(reps, 1, 1, 1)[:n_s].contiguous()
        long_out = torch.empty(n_s, 2, H, W, device="cuda")
        barrier()
        sampler2 = ClockSampler(local) if rank == 0 else None
        if sampler2:
            sampler2.start()
            time.sleep(0.12)
        t_s0 = time.perf_counter()
        e6, e7 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e6.record()
        ctx.colorize_clip(long_L, TEMPERATURE, out=long_out)
        e7.record()
        barrier()
        t_s1 = time.perf_counter()
        ms_s = max_over_ranks(e6.elapsed_time(e7))
        clk2 = sampler2.stop([(t_s0, t_s1)]) if sampler2 else None
        sustained = {"frames_per_gpu": n_s, "seconds": ms_s * 1e-3, "value": world * n_s / (ms_s * 1e-3), "unit": "frames/s",
                     "clocks": clk2, "note": "same leg as `value` (frames resident in HBM), run back to back for >= 2 s so "
                                             "that the chip reaches its power-limited steady state"}
        del long_L, long_out

    # ---------------- leg 3: per-kernel durations, one stream, no overlap (for the roofline objects) ----------------
    # The clip API overlaps two streams, so a kernel's event-bracketed time there includes its neighbours; the
    # roofline needs the kernel's own duration: same frames through dvc_colorize_frames on one stream, CUDA events
    # around every correlation / tensor-core convolution launch (on the launching stream), live in this run.
    KP = min(K, 5)
    last = torch.zeros(1, 3, H, W, device="cuda")
    ctx.colorize_frames(dev_L[0:1], last, TEMPERATURE)
    ctx.profile_corr(True)
    ctx.profile_conv(True)
    ctx.corr_mean_ms(True)
    ctx.conv_profile(0, reset=True)
    e4, e5 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e4.record()
    for t in range(Wm, Wm + KP):
        ab1 = ctx.colorize_frames(dev_L[t:t + 1], last, TEMPERATURE)
        last = torch.cat((dev_L[t:t + 1], ab1), 1)
    e5.record()
    torch.cuda.synchronize()
    ms_serial = e4.elapsed_time(e5) / KP
    corr_ms = ctx.corr_mean_ms(True)
    conv_all = ctx.conv_profile(0)
    conv_by = {v: ctx.conv_profile(v) for v in (256, 128, 64)}
    ctx.conv_profile(0, reset=True)
    ctx.profile_corr(False)
    ctx.profile_conv(False)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, ab=dev_out[K - 1:K])  # the value leg's last frame; no later leg writes dev_out

    peak, peak_src = measured_peak(ms_serial * KP * 1e-3)
    achieved = CORR_FLOP / (corr_ms * 1e-3) / 1e12 if corr_ms > 0 else 0.0
    conv_all_tflops = conv_all[2] / (conv_all[1] * 1e-3) / 1e12 if conv_all[1] > 0 else 0.0
    conv_detail = {str(v): {"launches_per_frame": n / KP, "ms_per_frame": ms / KP,
                            "tflops": (fl / (ms * 1e-3) / 1e12 if ms > 0 else 0.0)} for v, (n, ms, fl) in conv_by.items() if n}
    line = {
        "metric": METRIC, "value": world * K / (ms_dev * 1e-3), "unit": "frames/s", "n_gpus": world, "steps": K,
        "warmup": Wm, "ms_per_step": ms_dev / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {
            "workload": WORKLOAD,
            "N_positions": N_POS,
            "conv_math": ((f"tcgen05 {'3xFP16 on exactly scaled hi/lo planes' if args.tc_f16 else '3xTF32 operand split'}, "
                           f"{'CTA pairs (cta_group::2)' if args.tc_cluster == 2 else 'single CTAs'}, TMEM chunk = "
                           f"{args.tc_kc} k-block(s) promoted to fp32 registers")
                          if args.conv_math == "tf32x3" else "fp32 CUDA-core (two-level accumulation)"),
            "corr_math": args.corr_math,
            "weights": "seeded random (dvc/synth.py), no checkpoint available",
            "l2": "distinct frame per step; per-frame activation working set (>2 GB) exceeds the 126 MB L2",
            "exemplar_prepare_and_broadcast_ms": exemplar_ms,
        },
        "e2e": {"value": world * K / (ms_e2e * 1e-3), "unit": "frames/s", "h2d_bytes_per_step": H * W * 4,
                "d2h_bytes_per_step": 2 * H * W * 4},
        "gpu_launches": launches,
        "clocks": clocks,
        # dominant kernel by device time (profiles/launches_r2.md: conv_tc_kernel, all channel tiles, ~78 % of a frame; the
        # 128-channel tile alone ~50 %: the launcher moved the quarter-resolution 256-channel layers onto it)
        "roofline": {"kernel": "conv_tc_kernel (flat shifted GEMM on tcgen05, 3 MMA passes per product; all tensor-core convolution "
                               "launches of a frame, channel tiles 256 / 128 / 64 listed under other_variants)",
                     "bound": "tensor",
                     "achieved": conv_all_tflops, "peak": peak, "unit": "TFLOP/s", "frac": conv_all_tflops / peak if peak else None,
                     "traffic": ncu_traffic("conv_tc_kernel<128>"), "peak_source": peak_src,
                     "traffic_note": "DRAM bytes (read + write) of ONE profiled launch of the 128-channel tile, the largest class by "
                                     "device time (profiles/ncu_r2_traffic.json names the layer and its algorithmic bytes)",
                     "launches_per_frame": conv_all[0] / KP, "ms_per_frame": conv_all[1] / KP,
                     "note": "sum of algorithmic FLOPs (2 x output pixels x taps x Cin x Cout) / sum of CUDA-event launch times, "
                             "single-stream pass of %d frames inside this run; the 3 MMA passes of the operand split are not "
                             "counted, so frac is bounded by 1/3 of the dense 16-bit peak (cuBLAS itself reaches 66-76 %% of the "
                             "nominal 2.25 PFLOP/s on this chip: MEASURED_PEAKS.json)" % KP,
                     "other_variants": conv_detail},
        # the north-star kernel (BASELINE metric: correlation tensor-pipe fraction)
        "roofline_corr": {"kernel": (f"corr_screen_kernel + corr_rescore_kernel ({args.corr_math}, T<=2e-10: one fp16 pass locates every row's "
                                     "candidates within a rigorous error bound, exact fp32 re-scoring) incl. operand preparation"
                                     if (args.corr_screen and args.corr_math == "fp16x3") else
                                     f"corr_tc_kernel ({args.corr_math}) incl. operand split + merge"),
                          "bound": "tensor", "mma_passes": 1 if (args.corr_screen and args.corr_math == "fp16x3") else 3,
                          "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak if peak else None,
                          "traffic": ncu_traffic("corr_tc_kernel"), "peak_source": peak_src, "launch_ms": corr_ms,
                          "note": "algorithmic 2*N*N*(256+3) FLOP per launch (the reference's matmul + softmax + matmul) over the CUDA-event "
                                  "time of the whole launch sequence; the exact kernel spends 3 MMA passes per product (ceiling 1/3 of the "
                                  "dense 16-bit peak, 1/6 for tf32x3), the screened T->0 path one pass (ceiling 1; the shared-memory port "
                                  "allows ~128 B/clk = one pass at full rate)"},
        "serial_ms_per_frame": ms_serial,
        "rank_checksum": {"ok": rank_check_ok, "ranks": world,
                          "what": "bit pattern of ab for one common seeded frame, all_gather'ed and compared across ranks"},
        "clip64": clip64,
        "sustained": sustained,
        "conv_tc_all": {"launches_per_frame": conv_all[0] / KP, "ms_per_frame": conv_all[1] / KP,
                        "tflops": conv_all[2] / (conv_all[1] * 1e-3) / 1e12 if conv_all[1] > 0 else 0.0},
    }
    if args.cpu_sample > 0:
        tb = time.perf_counter()
        times, cores, _ = cpu_frames_per_sec(args.cpu_sample, warm=1)
        line["cpu_baseline"] = {"value": len(times) / sum(times), "unit": "frames/s", "cores": cores, "kind": "port",
                                "sample": f"{len(times)} frames of the same workload after 1 warm-up frame "
                                          f"({time.perf_counter() - tb:.0f} s of CPU work)"}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
