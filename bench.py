#!/usr/bin/env python
"""Headline benchmark: 4D-reconstruction frames/sec, 320x512x16f windows, 50-step DDIM, synthetic data.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--frames T] [--dump-outputs DIR]

One "step" = one full pass of the hot path over a FIXED synthetic clip (default 72 frames = 8 sliding windows of
16 frames, stride 8 -- the BASELINE.json configs[2]/[3] shape): per window VAE-encode of the 16 conditioning
frames -> 50 DDIM steps of the spatio-temporal U-Net (one CUDA graph per step) -> 4 VAE decodes (point map +
confidence, ray directions, ray moments, inverse depth) -> per-window post-processing; then the sliding-window
global alignment (init + 500 iterations in two persistent kernel launches + LAD / trajectory sub-alignments).
The clip is the same for every N (STRONG scaling): rank r diffuses the windows w with w % N == r, the per-window
predictions are all-gathered over NCCL/NVLink and the alignment runs SHARDED -- every rank optimises the depth
maps of its share of the images and the ranks exchange the reduced gradients inside the kernel, by stores into
peer memory.  `--frames 16` is BASELINE.json configs[1] (one window); the default run also times that
single-window case for a few steps and reports it under `single_window`.

`value` is timed with the video already in HBM; `e2e` includes the pinned-host -> device copy of every window's
frames and the device -> host read of depth maps / poses / focal every step.  `--impl reference` times the
reference's CPU path (its own modules when $GEO4D_REFERENCE names its source tree, else the oracle port) on a
bounded sample of the same workload, all host threads.

`--dump-outputs DIR` writes what the last timed step returned (see dump_outputs) so that two builds can be compared
output for output: every input -- weights, video, initial latents, the VAE posterior noise -- comes from a fixed
seed, so the same arguments give the same inputs in every run.  The GEMM tile autotuner picks by timing, and a
split-K choice changes rounding, which 50 DDIM steps and the alignment amplify; with GEO4D_AUTOTUNE=0 repeated
runs of one build give bit-identical outputs.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
import traceback

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

# algorithmic work, traced from the reference modules (SURVEY.md 2.2 / 8(d)), 2*MAC
UNET_TFLOP = {(320, 512): 12.61, (256, 256): 4.91, (576, 1024): 52.36}
VAE_TFLOP = {(320, 512): dict(dec=1.564, dec_conf=1.757, enc=0.690), (576, 1024): dict(dec=5.754, dec_conf=6.451, enc=2.609),
             (256, 256): dict(dec=0.622, dec_conf=0.700, enc=0.273)}


def peaks():
    p = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(bf16_burst=d["bf16_tflops"], bf16_sustained=d["bf16_tflops_sustained"], hbm=d["hbm_gbs"],
                    source="measured")
    return dict(bf16_burst=1590.0, bf16_sustained=1400.0, hbm=6650.0, source="fallback")


def committed_ncu():
    """Numbers only ncu can measure (DRAM bytes of one U-Net step, tensor-pipe activity of the attention kernel),
    read from the committed summary of the same tree -- labelled as such in the line, never timed here."""
    try:
        return json.load(open(os.path.join(REPO, "profiles", "r2_ncu_summary.json")))
    except Exception:
        return {}


def kernel_rooflines(dev, pk):
    """Live per-kernel numbers: every launch is timed GPU-bound (20 launches in a CUDA graph, CUDA events on the
    launching stream).  Tensor-bound kernels against the measured dense-bf16 burst peak, HBM-bound kernels
    (GroupNorm, the alignment iteration) against the measured copy bandwidth, both with ALGORITHMIC work
    (SURVEY.md 8(d): GN = one read + one write of the tensor; alignment = 28 B per (window, frame, pixel))."""
    import torch
    from geo4d_b200 import ops

    def gtime(fn, n=20):
        fn()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            g = torch.cuda.CUDAGraph()
            with ops.capture_graph(g):
                for _ in range(n):
                    fn()
            g.replay()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(side)
            for _ in range(3):
                g.replay()
            e1.record(side)
            e1.synchronize()
        torch.cuda.current_stream().wait_stream(side)
        return e0.elapsed_time(e1) * 1e-3 / (3 * n)

    bf = lambda *sh: torch.randn(*sh, device=dev).bfloat16()
    out = []

    def add(name, flops, sec, launches_per_step):
        ach = flops / sec * 1e-12
        out.append({"kernel": name, "bound": "tensor", "us": round(sec * 1e6, 2), "achieved": round(ach, 1),
                    "unit": "TFLOP/s", "peak": pk["bf16_burst"], "frac": round(ach / pk["bf16_burst"], 3),
                    "launches_per_unet_step": launches_per_step})

    def add_hbm(name, nbytes, sec, note):
        ach = nbytes / sec * 1e-9
        out.append({"kernel": name, "bound": "hbm", "us": round(sec * 1e6, 2), "achieved": round(ach, 1), "unit": "GB/s",
                    "peak": pk["hbm"], "frac": round(ach / pk["hbm"], 3), "algorithmic_bytes": nbytes, "note": note})

    x = bf(40960, 320); w9 = bf(9, 320, 320); b = torch.randn(320, device=dev); o = torch.empty(40960, 320, device=dev, dtype=torch.bfloat16)
    add("tap_gemm conv3x3 16x40x64 320->320", 2.0 * 40960 * 2880 * 320, gtime(lambda: ops.conv3x3(x, 16, 40, 64, w9, b, out=o)), 7)
    x1 = bf(10240, 640); w1 = bf(9, 640, 640); b1 = torch.randn(640, device=dev); o1 = torch.empty(10240, 640, device=dev, dtype=torch.bfloat16)
    add("tap_gemm conv3x3 16x20x32 640->640", 2.0 * 10240 * 5760 * 640, gtime(lambda: ops.conv3x3(x1, 16, 20, 32, w1, b1, out=o1)), 6)
    x3 = bf(640, 1280); w3 = bf(9, 1280, 1280); b3 = torch.randn(1280, device=dev); o3 = torch.empty(640, 1280, device=dev, dtype=torch.bfloat16)
    add("tap_gemm conv3x3 16x5x8 1280->1280", 2.0 * 640 * 11520 * 1280, gtime(lambda: ops.conv3x3(x3, 16, 5, 8, w3, b3, out=o3)), 8)
    wl = bf(320, 320)
    add("tap_gemm linear 40960x320->320 (+bias)", 2.0 * 40960 * 320 * 320, gtime(lambda: ops.linear(x, wl, b, out=o)), 45)
    wg = bf(2560, 320); bg = torch.randn(2560, device=dev); og = torch.empty(40960, 1280, device=dev, dtype=torch.bfloat16)
    add("tap_gemm linear 40960x320->2560 GEGLU", 2.0 * 40960 * 320 * 2560, gtime(lambda: ops.linear(x, wg, bg, act=ops.ACT_GEGLU, out=og)), 10)
    qkv = bf(40960, 960)
    add("attn_fwd B16 H5 L2560 d64", 4.0 * 16 * 5 * 2560 * 2560 * 64,
        gtime(lambda: ops.attention(qkv[:, :320], qkv[:, 320:640], qkv[:, 640:], o, 16, 5, 2560, 2560)), 5)
    qkv1 = bf(10240, 1920)
    add("attn_fwd B16 H10 L640 d64", 4.0 * 16 * 10 * 640 * 640 * 64,
        gtime(lambda: ops.attention(qkv1[:, :640], qkv1[:, 640:1280], qkv1[:, 1280:], o1, 16, 10, 640, 640)), 10)
    kvt = bf(77, 640)
    add("attn_fwd cross B16 H5 Lq2560 Lk77 (text)", 4.0 * 16 * 5 * 2560 * 77 * 64,
        gtime(lambda: ops.attention(qkv[:, :320], kvt[:, :320], kvt[:, 320:], o, 16, 5, 2560, 77, kv_batch_div=16)), 5)
    g32 = torch.ones(320, device=dev); be = torch.zeros(320, device=dev)
    add_hbm("gn_fused_kernel GroupNorm+SiLU 16x(2560 rows) C=320", 2 * 40960 * 320 * 2,
            gtime(lambda: ops.groupnorm(x, 16, 2560, g32, be, 1e-5, True, out=o)), "read + write of the bf16 tensor")
    return out


def align_roofline(dev, pk, H, W):
    """One window (16 images, 320x512) through the persistent alignment loop: 100 iterations in one launch."""
    import torch
    from geo4d_b200.cloud_opt import LightPointCloudGroupOptimizer
    T, HW = 16, H * W
    g = torch.Generator(device=dev).manual_seed(5)
    pts = torch.randn(T, H, W, 3, device=dev, generator=g) + torch.tensor([0.0, 0.0, 4.0], device=dev)
    pred = {"pts3d": pts, "conf": 1 + torch.rand(T, H, W, 1, device=dev, generator=g),
            "inverse_depthmap": 0.1 + torch.rand(T, H, W, 1, device=dev, generator=g),
            "traj": torch.eye(4, device=dev).repeat(T, 1, 1)}
    views = [[{"idx": (i,)} for i in range(T)]]
    sc = LightPointCloudGroupOptimizer(views, [pred], conf="id", conf_optimize=True, verbose=False, shared_focal=True,
                                       num_total_iter=100, temporal_smoothing_weight=0.015, translation_weight=1.0,
                                       depth_traj_start_iter=100, shard_alignment=False, engine="loop")
    with torch.no_grad():
        sc.im_depthmaps.fill_(1.4)
    best = None
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        sc._global_alignment_loop(lr=0.03, niter=100, schedule="linear", lr_min=1e-3)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        best = ms if best is None else min(best, ms)
    sec = best * 1e-3 / 100
    nbytes = 28 * T * HW
    return {"kernel": "align_loop_kernel (per iteration, 1 window = 16 images)", "bound": "hbm", "us": round(sec * 1e6, 2),
            "achieved": round(nbytes / sec * 1e-9, 1), "unit": "GB/s", "peak": pk["hbm"],
            "frac": round(nbytes / sec * 1e-9 / pk["hbm"], 3), "algorithmic_bytes": nbytes,
            "note": "28 B per (window, frame, pixel) (SURVEY 8(d)); the 115 MB working set is L2-resident, "
                    "includes 2 grid barriers + the small-parameter step per iteration"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active") and not v.lower().startswith("not"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def n_windows_of(T):
    from geo4d_b200.pipeline import sliding_windows
    return len(sliding_windows(T, 8))


DUMP_MAX_PIXELS = 1 << 22   # per-pixel arrays of larger clips are sampled: 2 x 16 MB, well under 64 MB in all


def dump_outputs(scene, out_dir):
    """The arrays a caller of the timed path receives from the aligned scene, as out_dir/<name>.npy (float32):
    depth maps and confidence [T, H, W], camera-to-world poses [T, 4, 4], focals [T, 1], principal points [T, 2].
    When the clip has more than DUMP_MAX_PIXELS pixels, depth and confidence are taken at one fixed seeded sample
    of pixel indices (sorted, flattened over T, H, W), the same in every run with the same clip shape."""
    import numpy as np
    import torch
    depth = torch.stack(scene.get_depthmaps())
    conf = torch.stack(scene.get_conf())
    if depth.numel() > DUMP_MAX_PIXELS:
        idx = torch.randperm(depth.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_MAX_PIXELS]
        idx = idx.sort().values.to(depth.device)
        depth, conf = depth.reshape(-1)[idx], conf.reshape(-1)[idx]
    out = {"depthmaps": depth, "conf": conf, "poses": scene.get_im_poses(), "focals": scene.get_focals(),
           "principal_points": scene.get_principal_points()}
    os.makedirs(out_dir, exist_ok=True)
    for name, t in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())


# ----------------------------------------------------------------------------------------------- reference arm
def _reference_modules():
    """The reference's own U-Net / VAE classes when its tree is importable ($GEO4D_REFERENCE, or baseline/_ref in
    this tree), else None -> the oracle port."""
    for root in (os.environ.get("GEO4D_REFERENCE"), os.path.join(REPO, "baseline", "_ref")):
        if root and os.path.isdir(os.path.join(root, "lvdm", "modules", "networks")):
            try:
                sys.path.insert(0, root)
                from oracle.gen_golden import install_shims
                install_shims()
                from lvdm.modules.networks.openaimodel3d import UNetModel
                from lvdm.modules.networks.ae_modules import Encoder, Decoder
                return dict(root=root, UNetModel=UNetModel, Encoder=Encoder, Decoder=Decoder)
            except Exception:
                if root in sys.path:
                    sys.path.remove(root)
    return None


def run_reference(args, rank, world, quiet=False):
    """CPU baseline on a bounded sample of the same workload, fp32 PyTorch on the host threads:
    ONE U-Net step of a full 16-frame window (temporal_length = 16, so temporal attention / temporal convolutions
    do real work) at 64x128, one frame through each VAE pass at 128x256, and a 24-image alignment (3 windows,
    64x96, init + 8 iterations).  Extrapolated linearly in pixels / steps / frames / windows / iterations to the
    workload (the quadratic spatial attention makes the linear pixel extrapolation favour the CPU arm)."""
    if rank != 0:
        return None
    import math
    import torch
    from oracle import unet as ou, vae as ov, align as oa
    H, W, T = args.height, args.width, args.frames
    n_windows = n_windows_of(T)
    cores = min(os.cpu_count() or 1, 32)   # OpenMP teams beyond 32 threads spend their time in fork/join on these operators
    torch.set_num_threads(cores)
    torch.set_flush_denormal(True)
    ref = _reference_modules()
    kind = "reference" if ref is not None else "port"
    Hs, Ws = 64, 128            # U-Net sample: 16 frames, latents 8x16
    Hv, Wv = 128, 256           # VAE sample: one frame
    g = torch.Generator().manual_seed(0)
    _base = torch.randn(1 << 25, generator=torch.Generator().manual_seed(7))
    _scaled = {}

    def cheap_params(shapes):
        # 1.4e9 weights: every weight is a read-only VIEW into one 32M-sample normal block pre-scaled to ~1/sqrt(fan_in)
        # (timing does not depend on the values as long as activations stay well scaled); norm gains 1, biases 0
        out, off = {}, 0
        for name, shp in shapes.items():
            n = 1
            for d in shp:
                n *= int(d)
            if len(shp) == 1:
                out[name] = torch.ones(shp) if name.endswith("weight") else torch.zeros(shp)
                continue
            fan = max(1, n // max(1, int(shp[0])))
            k = max(0, int(round(math.log2(fan))))
            if k not in _scaled:
                _scaled[k] = _base * (2.0 ** (-k / 2))
            blk = _scaled[k]
            assert n <= blk.numel(), (name, shp)
            off = ((off + 7919 * 64) % (blk.numel() - n + 1)) // 64 * 64      # 256-byte aligned views
            out[name] = blk[off:off + n].view(shp)
        return out

    cfg = ou.UNetConfig(temporal_length=16)
    sd = cheap_params(ou.param_shapes(cfg))
    x = torch.randn(1, 20, 16, Hs // 8, Ws // 8, generator=g)
    ctx = torch.randn(1, 77 + 16 * 16, 1024, generator=g)
    ts = torch.tensor([499])
    fs = torch.tensor([24])
    vcfg = ov.VAEConfig()
    vsd = cheap_params(ov.param_shapes(vcfg))
    z = torch.randn(1, 4, Hv // 8, Wv // 8, generator=g)
    img = torch.randn(1, 3, Hv, Wv, generator=g)
    unet_fn = lambda: ou.forward(cfg, sd, x, ts, ctx, fs)
    if ref is not None:
        try:   # the reference's own module on the same weights (meta construction + assign: no 6 GB re-initialisation)
            import yaml
            ycfg = yaml.safe_load(open(os.path.join(REPO, "configs", "inference_geo4d.yaml")))
            up = dict(ycfg["model"]["params"]["unet_config"]["params"])
            up["use_checkpoint"] = False
            with torch.device("meta"):
                net = ref["UNetModel"](**up)
            net.load_state_dict(sd, strict=True, assign=True)
            net.eval()
            unet_fn = lambda: net(x, ts, context=ctx, fs=fs)
        except Exception as ex:
            kind = "port"
            if not quiet:
                print(f"[bench] reference modules not usable ({type(ex).__name__}: {ex}); timing the oracle port", file=sys.stderr)

    def timed(fn):
        t0 = time.time()
        with torch.no_grad():
            fn()
        return time.time() - t0

    with torch.no_grad():   # one untimed pass of everything (thread pool, primitive caches, page faults)
        unet_fn()
        ov.decode_with_conf_adaptor(vcfg, vsd, z); ov.decode(vcfg, vsd, z); ov.encode_moments(vcfg, vsd, img)
    reps = max(1, min(args.steps, 2))
    t_unet = sum(timed(unet_fn) for _ in range(reps)) / reps * (H * W) / float(Hs * Ws)          # per window step
    pxv = (H * W) / float(Hv * Wv)
    t_dc = timed(lambda: ov.decode_with_conf_adaptor(vcfg, vsd, z)) * pxv
    t_d = timed(lambda: ov.decode(vcfg, vsd, z)) * pxv
    t_e = timed(lambda: ov.encode_moments(vcfg, vsd, img)) * pxv
    # alignment sample: 24 images (3 windows) at 64x96: initialisation + 8 iterations, per (image, pixel, iteration)
    Ta, Ha, Wa, its = 24, 64, 96, 8
    groups, preds, _ = oa.synthetic_scene(T=Ta, H=Ha, W=Wa, noise=0.003)
    al = oa.GroupAligner(groups, preds, depth_traj_start_iter=10 ** 6, lad_max_iters=10)
    t0 = time.time(); al.init_from_group(10); t_init = time.time() - t0
    t0 = time.time(); al.compute_global_alignment(niter=its, lr=0.03, schedule="linear"); t_loop = max(time.time() - t0 - t_init, 1e-6)
    edges = n_windows * 16
    scale_px = (H * W) / float(Ha * Wa)
    t_align = t_init * scale_px * edges / (len(groups) * 16) + (t_loop / its) * args.align_iters * scale_px * edges / (len(groups) * 16)
    window_s = args.ddim_steps * t_unet + 16 * (t_dc + 3 * t_d) + 16 * t_e
    total_s = window_s * n_windows + t_align
    value = T / total_s
    sample = (f"{kind}: 1 U-Net step of a 16-frame window (temporal_length 16) at {Hs}x{Ws}; 1 decode+conf, 1 plain decode, "
              f"1 encode of one frame at {Hv}x{Wv}; alignment init + {its} iterations of {Ta} images at {Ha}x{Wa} "
              f"(LAD fit excluded); fp32 PyTorch on {cores} threads; extrapolated linearly to {H}x{W}, {args.ddim_steps} "
              f"steps, 16 frames x {n_windows} window(s), {args.align_iters} alignment iterations")
    line = {"impl": "reference", "metric": "4D-recon frames/sec", "value": value, "unit": "frames/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": total_s * 1e3,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{T}f {H}x{W}, {args.ddim_steps}-step DDIM, {n_windows} window(s) stride 8, "
                                   f"{args.align_iters}-iter alignment", "extrapolated": True},
            "cpu_baseline": {"value": value, "unit": "frames/s", "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "phases_s": {"unet_step_window": t_unet, "decode_conf_frame": t_dc, "decode_frame": t_d, "encode_frame": t_e,
                         "alignment": t_align}}
    if not quiet:
        print(json.dumps(line))
    return line


# ----------------------------------------------------------------------------------------------- B200 arm
def run_b200(args, rank, world, local):
    import torch
    import torch.distributed as dist
    from geo4d_b200 import ops, sharding, synthetic
    from geo4d_b200.pipeline import Geo4DPipeline, sliding_windows
    torch.cuda.set_device(local)
    # the VAE encoder draws its posterior noise from the global CPU generator, which torch does not seed the same
    # way in every process: seeded here, every run with the same arguments gets the same inputs
    torch.manual_seed(0)
    dev = torch.device("cuda", local)
    if world > 1:
        import datetime
        # a rank that dies or diverges must not leave the others blocked for NCCL's default 10 minutes
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=300))
    H, W, T = args.height, args.width, args.frames
    model, pm_vae, cfg = synthetic.build_model(device=dev, seed=0)
    pipe = Geo4DPipeline(model, pm_vae, ddim_steps=args.ddim_steps, postprocess=dict(cfg["postprocess"], silent=True,
                                                                                     n_iter=args.align_iters))
    windows = sliding_windows(T, 8)
    n_win = len(windows)
    mine = sharding.windows_for_rank(n_win, rank, world)
    video_host = synthetic.synthetic_video(T, H, W, device="cpu", seed=123)
    host_win = {w: video_host[:, :, windows[w]].contiguous().pin_memory() for w in mine}
    dev_win = {w: host_win[w].to(dev, non_blocking=True) for w in mine}
    views = [[{"idx": (i,)} for i in range(w.start, w.stop)] for w in windows]
    one = [slice(0, 16, 1)]

    def step(win_video):
        """this rank's windows -> predictions -> (all-gather) -> sharded global alignment; returns the scene"""
        local_preds = {}
        for w in mine:
            xt = torch.randn((1, 16, 16, H // 8, W // 8), device=dev, generator=torch.Generator(device=dev).manual_seed(123 + w))
            _, preds = pipe.reconstruct(win_video[w], stride=8, windows=one, align=False, x_T_fn=lambda wi: xt)
            local_preds[w] = preds[0]
        with pipe.phase("gather"):
            preds = sharding.gather_predictions(local_preds, n_win, 16, H, W)
        with torch.enable_grad():
            scene = pipe.post_optimization(views, preds)
        return scene

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step(dev_win)
    # ---- timed region 1: device-resident input
    barrier()
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    n0 = ops.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    pipe.events = []
    e0.record()
    for _ in range(args.steps):
        scene = step(dev_win)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    launches = ops.launch_count() - n0
    phase_ms = pipe.phase_ms()
    shard_info = getattr(scene, "_shard", None)
    if args.dump_outputs and rank == 0:
        dump_outputs(scene, args.dump_outputs)
    # ---- timed region 2: end to end from pinned host memory, results read back (fewer steps: same per-step work)
    e2e_steps = max(1, min(args.steps, args.e2e_steps if args.e2e_steps > 0 else max(2, args.steps // 4)))
    barrier()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record()
    d2h = 0
    for _ in range(e2e_steps):
        vd = {w: host_win[w].to(dev, non_blocking=True) for w in mine}
        sc = step(vd)
        if rank == 0:
            outs = [torch.stack(sc.get_depthmaps()).cpu(), sc.get_im_poses().detach().cpu(), sc.get_focals().detach().cpu()]
            d2h = sum(o.numel() * o.element_size() for o in outs)
    e3.record()
    barrier()
    ms_e2e = e2.elapsed_time(e3)
    clk = clocks.stop() if rank == 0 else None
    t = torch.tensor([ms, ms_e2e], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_e2e = float(t[0]), float(t[1])
    if rank != 0:
        if world > 1:
            dist.barrier()   # rank 0 still uses the GPU for the per-kernel rows; leave together
            dist.destroy_process_group()
        return
    pk = peaks()
    ncu = committed_ncu()
    n_mine = max(1, len(mine))
    unet_ms = phase_ms.get("ddim", 0.0) / max(1, args.steps * args.ddim_steps * n_mine)
    tflop = UNET_TFLOP.get((H, W))
    roof = None
    if tflop and unet_ms > 0:
        ach = tflop / (unet_ms * 1e-3)
        roof = {"bound": "tensor", "kernel": "U-Net step (1 CUDA-graph launch; tap_gemm_kernel = 93% of its FLOPs)",
                "achieved": ach, "peak": pk["bf16_sustained"], "unit": "TFLOP/s", "frac": ach / pk["bf16_sustained"],
                "peak_source": pk["source"] + " (sustained: timed inside a long step)",
                "traffic": ncu.get("unet_step_dram_bytes"),
                "traffic_source": "ncu dram__bytes_read+write of one U-Net step, committed pass profiles/r2_ncu_summary.json"
                                  if ncu.get("unet_step_dram_bytes") else None,
                "algorithmic_tflop_per_launch": tflop, "ms_per_launch": unet_ms}
        try:
            roof["kernels"] = kernel_rooflines(dev, pk)
            roof["kernels"].append(align_roofline(dev, pk, H, W))
        except Exception as ex:  # pragma: no cover
            roof["kernels_error"] = repr(ex)
        vt = VAE_TFLOP.get((H, W))
        if vt and phase_ms.get("decode", 0) > 0:
            dec_ms = phase_ms["decode"] / (args.steps * n_mine)
            enc_ms = phase_ms.get("encode", 0.0) / (args.steps * n_mine)
            roof["vae"] = {"decode_ms_per_window": dec_ms, "decode_tflops": 16 * (vt["dec_conf"] + 3 * vt["dec"]) / (dec_ms * 1e-3),
                           "encode_ms_per_window": enc_ms, "encode_tflops": (16 * vt["enc"] / (enc_ms * 1e-3)) if enc_ms else None}
    # attention tensor-pipe utilisation (second half of BASELINE.json:metric): live = achieved attention FLOP/s of the
    # L = 2560 kernel / measured dense bf16 burst peak; ncu = sm__pipe_tensor_cycles_active of the same kernel from
    # the committed ncu --set full capture of this tree
    attn_pct = None
    if roof and roof.get("kernels"):
        for k in roof["kernels"]:
            if k["kernel"].startswith("attn_fwd B16 H5 L2560"):
                attn_pct = {"live_flop_based_pct": round(100.0 * k["frac"], 1), "achieved_tflops": k["achieved"],
                            "ncu_pipe_tensor_cycles_active_pct": ncu.get("attn_L2560_pipe_tensor_pct"),
                            "ncu_source": "profiles/r2_ncu_summary.json" if ncu.get("attn_L2560_pipe_tensor_pct") is not None else None}
    value = T * args.steps / (ms * 1e-3)
    h2d = n_win * 16 * 3 * H * W * 4
    line = {"metric": "4D-recon frames/sec", "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": f"{T}f {H}x{W}, {args.ddim_steps}-step DDIM (cfg 1, eta 0, uniform_trailing), "
                                   f"{n_win} window(s) of 16f stride 8, {args.align_iters}-iter alignment; the same clip for every N",
                       "l2": "weights 2.9 GB + activations >> 126 MB L2 (no flush needed)",
                       "weights": "seeded synthetic", "parallelism": f"window-parallel x{world} ({len(mine)} window(s) on rank 0), "
                                                                     f"alignment {'sharded ' + str(shard_info) if shard_info and shard_info.get('world', 1) > 1 else 'on one GPU'}",
                       "gemm_autotune": f"{len(ops.tuned_configs())} shapes pinned during warm-up"},
            "e2e": {"value": T * e2e_steps / (ms_e2e * 1e-3), "unit": "frames/s", "steps": e2e_steps,
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": launches, "clocks": clk, "roofline": roof, "attn_tensor_pipe_pct": attn_pct,
            "phases_ms_per_step": {k: v / args.steps for k, v in phase_ms.items()}}
    # ---- BASELINE.json configs[1]: the single-window case on this GPU, a few steps (device-resident input)
    if T != 16 and args.single_window_steps > 0:
        try:
            v16 = synthetic.synthetic_video(16, H, W, device=dev, seed=123)

            def step16():
                sc, _ = pipe.reconstruct(v16, stride=8, x_T_fn=lambda wi: torch.randn(
                    (1, 16, 16, H // 8, W // 8), device=dev, generator=torch.Generator(device=dev).manual_seed(123)))
                return sc
            old_shard = os.environ.get("GEO4D_ALIGN_SHARD")
            os.environ["GEO4D_ALIGN_SHARD"] = "0"   # rank 0 alone runs this case
            for _ in range(2):
                step16()
            torch.cuda.synchronize()
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            pipe.events = []
            a0.record()
            for _ in range(args.single_window_steps):
                step16()
            a1.record()
            torch.cuda.synchronize()
            ms16 = a0.elapsed_time(a1) / args.single_window_steps
            line["single_window"] = {"workload": f"16f {H}x{W}, {args.ddim_steps} steps, 1 window + {args.align_iters}-iter alignment "
                                                 "(BASELINE.json configs[1]), 1 GPU", "frames_per_s": 16 / (ms16 * 1e-3),
                                     "ms_per_step": ms16, "steps": args.single_window_steps,
                                     "phases_ms_per_step": {k: v / args.single_window_steps for k, v in pipe.phase_ms().items()}}
            if old_shard is None:
                os.environ.pop("GEO4D_ALIGN_SHARD", None)
            else:
                os.environ["GEO4D_ALIGN_SHARD"] = old_shard
        except Exception as ex:  # pragma: no cover
            line["single_window"] = {"error": repr(ex)}
    if not args.no_cpu_baseline:
        try:
            ref = run_reference(argparse.Namespace(**{**vars(args), "steps": 1, "warmup": 0}), 0, world, quiet=True)
            line["cpu_baseline"] = ref["cpu_baseline"]
        except Exception as ex:  # pragma: no cover
            line["cpu_baseline"] = {"error": repr(ex)}
    print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--height", type=int, default=320)
    ap.add_argument("--width", type=int, default=512)
    ap.add_argument("--frames", type=int, default=72, help="clip length; 72 = 8 windows of 16 frames, stride 8")
    ap.add_argument("--ddim-steps", type=int, default=50)
    ap.add_argument("--align-iters", type=int, default=500)
    ap.add_argument("--e2e-steps", type=int, default=0, help="steps of the end-to-end region (0: max(2, steps/4))")
    ap.add_argument("--single-window-steps", type=int, default=3)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (float32, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    try:
        if args.impl == "reference":
            run_reference(args, rank, world)
        else:
            run_b200(args, rank, world, local)
    except Exception as ex:
        # a failing rank must say why: the traceback on stderr and, from rank 0, a final JSON line
        sys.stderr.write(f"[bench rank {rank}] FAILED\n{traceback.format_exc()}\n")
        sys.stderr.flush()
        if rank == 0:
            print(json.dumps({"error": f"{type(ex).__name__}: {ex}", "rank": rank, "n_gpus": world,
                              "traceback_tail": traceback.format_exc().strip().splitlines()[-6:]}))
            sys.stdout.flush()
        sys.exit(1)


if __name__ == "__main__":
    main()
