#!/usr/bin/env python
"""Benchmark of the STAR denoising hot path on B200 (driver contract: one JSON line on rank 0).

Metric (BASELINE.json): upscaled frames/sec, 4x 240p->960p I2VGen-XL, 32-frame chunks, 50 steps.
  * workload (N=1): BASELINE.json configs[1] -- one 32-frame chunk at latent 122x216 (240p -> 960p
    after pad_to_fit, 976x1728 px), default ControlledV2VUNet (2.04 B parameters, synthetic non-zero
    weights), CFG 7.5 (2 UNet+ControlNet forwards per solver step), dpmpp_2m_sde 'normal' schedule.
  * a "step" = ONE solver step of that schedule = 2 forwards + guidance + solver update.
  * value = chunk frames / (50 * mean step time): frames per second of the full 50-step denoise.  The VAE legs
    (star_b200's temporal VAE, parity unpinned) are timed separately and reported under `pipeline`.
  * N>1: one 32-frame chunk per GPU of a single F=16(N+1)-frame clip (stride 16, as make_chunks
    produces), exact per-step x0 all-gather (diffusion_sdedit.sample_sr).  The unit of work is the
    32-frame chunk the metric names: value = 32 N chunk-frames / time ("scaling": "weak", one chunk per
    GPU).  Neighbouring chunks overlap by 16 frames and the reference re-computes the overlap on every
    chunk, so the clip has 16(N+1) unique frames: that rate is config.unique_frames_per_s.
  * e2e: the same metric through VideoToVideo_sr.denoise_latents() from pinned HOST tensors, one
    1-step call per "step": H2D of latent + text embeddings and D2H of the result inside the timing.
  * gpu_reference (N=1): the UNMODIFIED reference modules (.half() + autocast, xformers -> SDPA) timed on the same B200 on
    the same shape in a child process (tools/ref_gpu.py; needs the staged tree oracle/_ref, see oracle/stage_reference.py):
    the denominator of the north-star's ">= 8x the reference's single-GPU PyTorch frames/sec".
  * config3 (N>=6): BASELINE config 3 -- a 72-frame clip = chunks 32/32/40 -- on the same ranks with the CFG-branch split
    (6 active ranks, load imbalance 40/32), reported beside the weak-scaling line.
  * --impl reference: the oracle's CPU/fp32 restatement of the reference path (oracle/unet_ref.py,
    pinned against the real reference) timed on the host cores on a bounded sample.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

LAT_H, LAT_W, CHUNK = 122, 216, 32
SCHEDULE_STEPS = 50
METRIC = "upscaled frames/sec, 4x 240p->960p I2VGen-XL, 32-frame chunks, 50 steps"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="star", choices=["star", "reference"])
    ap.add_argument("--lat-h", type=int, default=LAT_H)
    ap.add_argument("--lat-w", type=int, default=LAT_W)
    ap.add_argument("--frames", type=int, default=0, help="override clip length (default 32, or 16(N+1) for N>1)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-reference", action="store_true", help="skip the reference-on-this-GPU block (needs oracle/_ref)")
    ap.add_argument("--trace-out", default="", help="write the per-op time table of the timed region to this file")
    ap.add_argument("--no-vae", action="store_true", help="skip the (separately reported) VAE encode/decode legs")
    ap.add_argument("--small", action="store_true", help="reduced model (debug only; not a valid bench line)")
    ap.add_argument("--workload", default="denoise", choices=["denoise", "vae", "cogvideox"],
                    help="denoise = BASELINE config 2 (the driver's line); vae = config 5 decode sweep; cogvideox = config 4 DiT step")
    ap.add_argument("--lib", default="", help="A/B: load this variant of libstar_sm100.so (tools/build_variant.py); not a valid bench line")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write what the last timed call returned (the denoised latent) to DIR/<name>.npy, float32: the seeded "
                         "inputs and weights make it comparable output for output between two builds run with the same arguments")
    return ap.parse_args()


DUMP_BYTES = 64 << 20


def dump_outputs(dirname, arrays):
    """{name: tensor} -> DIR/<name>.npy in float32, at most DUMP_BYTES in all: a larger output is replaced by a fixed, seeded
    sample of its elements (same positions in every run), stored flat as <name>.sample.npy."""
    os.makedirs(dirname, exist_ok=True)
    per = DUMP_BYTES // max(1, len(arrays)) // 4
    for name, t in arrays.items():
        t = t.detach().float()
        if t.numel() > per:
            idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:per].to(t.device)
            t, name = t.reshape(-1)[idx], name + ".sample"
        np.save(os.path.join(dirname, name + ".npy"), t.cpu().numpy())


def solver_steps(steps, total_noise_levels=1000):
    """solver steps diffusion_sdedit.sample_sr runs for an int `steps` with dpmpp_2m_sde on the 'trailing' grid: it builds
    steps + 1 timesteps with a float arange and drops the penultimate one, and for a few counts (60, 102, 120, ...) the arange
    rounds up to one timestep more."""
    return len(torch.arange(total_noise_levels - 1, -1, -(total_noise_levels / (steps + 1)))) - 1


# ---------------------------------------------------------------------------------- helpers
class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx = float(r[2])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        d = json.load(open(p))
        return {"tflops": d.get("bf16_tflops_sustained", d.get("bf16_tflops")), "hbm_gbs": d.get("hbm_gbs"),
                "source": "MEASURED_PEAKS.json (bf16_tflops_sustained: kernel timed inside a long step)"}
    return {"tflops": 1590.0, "hbm_gbs": 6650.0, "source": "fallback (B200_PROFILING.md)"}


def ncu_traffic_bytes():
    """DRAM bytes per launch of the dominant kernel from the committed ncu --set full capture (profiles/)."""
    path = os.path.join(ROOT, "profiles", "r02_ncu_attn4.txt")
    if not os.path.isfile(path):
        path = os.path.join(ROOT, "profiles", "r01_ncu_attn4_split.txt")
    if not os.path.isfile(path):
        return None
    mult = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    tot = 0.0
    for line in open(path):
        parts = line.split()
        if len(parts) >= 3 and parts[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum") and parts[1] in mult:
            tot += float(parts[2]) * mult[parts[1]]
    return tot or None


def build_model(small, device, seed=2, on_cpu_first=False):
    from star_b200.utils.synth import synth_state_dict
    from star_b200.video_to_video.modules.unet_v2v import ControlledV2VUNet
    kw = dict(dim_mult=[1, 2, 1, 4], num_res_blocks=1) if small else {}
    with torch.device("meta"):
        net = ControlledV2VUNet(**kw)
    manifest = {k: tuple(v.shape) for k, v in net.state_dict().items()}
    sd = synth_state_dict(manifest, seed=seed, device="cpu" if on_cpu_first else device)
    net.load_state_dict({k: v.to(device, torch.float16) for k, v in sd.items()}, assign=True)
    net.eval()
    return net, (sd if on_cpu_first else None), kw


def synth_inputs(F, H, W, seed=0):
    g = torch.Generator().manual_seed(seed)
    feat = 0.5 * torch.randn(1, 4, F, H, W, generator=g)
    y = torch.randn(1, 77, 1024, generator=g)
    ny = torch.randn(1, 77, 1024, generator=g)
    return feat, y, ny


class _StubText:
    """Text embeddings are inputs of the hot path (north_star); the OpenCLIP tower is out of scope."""

    def __init__(self, emb):
        self.emb = emb

    def __call__(self, s):
        return self.emb


# ---------------------------------------------------------------------------------- CPU reference arm
# The reference's CPU path is ~1e4 x slower than the GPU path (one fp32 forward of ONE frame at latent 122x216
# takes ~220 s on 128 host cores), so it is timed on a bounded sample -- 1 frame at latent 34x64 -- and
# extrapolated by ALGORITHMIC FLOPs counted with the same counter (torch.utils.flop_counter) on the sample and,
# on meta tensors, on the full workload: frames/s = frames / (steps * flops_full_step / measured_flop_rate).
CPU_SAMPLE = (1, 34, 64)         # frames, latent H (2 mod 8), latent W (0 mod 8)


def cpu_threads():
    """threads for the CPU arm: all cores up to 32 (the bounded sample is too small to scale further; more threads
    only add synchronisation overhead on the 128-core hosts of this pool)"""
    return max(1, min(os.cpu_count() or 1, int(os.environ.get("STAR_CPU_THREADS", "32"))))


def oracle_flops(kw, frames, H, W):
    """algorithmic FLOPs (2*MAC, attention 4*Nq*Nk*d) of ONE oracle forward, counted on meta tensors"""
    from torch.utils.flop_counter import FlopCounterMode
    from oracle.unet_ref import UNetCfg, controlled_unet_forward
    from star_b200.video_to_video.modules.unet_v2v import ControlledV2VUNet
    with torch.device("meta"):
        net = ControlledV2VUNet(**kw)
        sd = {k: torch.empty(v.shape) for k, v in net.state_dict().items()}
        x = torch.empty(1, 4, frames, H, W)
        y = torch.empty(1, 77, 1024)
        t = torch.zeros(1, dtype=torch.long)
    with FlopCounterMode(display=False) as fc:
        controlled_unet_forward(sd, x, t, y, x, UNetCfg(**kw))
    return float(fc.get_total_flops())


def cpu_sample_setup(kw):
    from star_b200.utils.synth import synth_state_dict
    from star_b200.video_to_video.modules.unet_v2v import ControlledV2VUNet
    with torch.device("meta"):
        net = ControlledV2VUNet(**kw)
    return synth_state_dict({k: tuple(v.shape) for k, v in net.state_dict().items()}, seed=2)


def cpu_step_fn(sd, kw, sample):
    """(step(), kind): one solver step of the reference path on the host cores.  kind "reference" = the reference's OWN, unmodified
    modules (oracle/ref_loader: /root/reference in the build container, the staged oracle/_ref on a GPU box); kind "port" = the
    pinned CPU restatement oracle/unet_ref.py (reduced debug model, or no reference tree on this machine)."""
    fs, H, W = sample
    feat, y, ny = synth_inputs(fs, H, W, seed=1)
    x = torch.randn(1, 4, fs, H, W)
    t = torch.tensor([899])
    net = None
    if not kw:
        try:
            from oracle.ref_loader import build_reference_unet, reference_available
            if reference_available():
                net = build_reference_unet(state_dict=sd)
        except Exception:
            net = None
    if net is not None:
        def step():                  # diffusion_sdedit.py:81,88-97: two model calls + guidance combine
            with torch.no_grad():
                a = net(x, t, y, hint=feat)
                b = net(x, t, ny, hint=feat)
                return b + 7.5 * (a - b)
        return step, "reference"
    from oracle.unet_ref import UNetCfg, controlled_unet_forward

    def step():                      # one solver step on the sample: 2 CFG forwards + guidance combine
        a = controlled_unet_forward(sd, x, t, y, feat, UNetCfg(**kw))
        b = controlled_unet_forward(sd, x, t, ny, feat, UNetCfg(**kw))
        return b + 7.5 * (a - b)
    return step, "port"


def cpu_extrapolate(dt_step, kw, sample, H, W):
    """seconds per solver step on the sample -> frames/s of the full CHUNK-frame, HxW workload"""
    f_sample = 2.0 * oracle_flops(kw, *sample)
    f_full = 2.0 * oracle_flops(kw, CHUNK, H, W)
    rate = f_sample / dt_step                                   # FLOP/s the host sustains on this path
    value = CHUNK / (SCHEDULE_STEPS * f_full / rate)
    note = (f"sample = one solver step (2 CFG forwards) of {sample[0]} frame(s) at latent {sample[1]}x{sample[2]}, fp32: "
            f"{dt_step:.2f} s = {rate / 1e12:.3f} TFLOP/s; full step = {f_full / 1e12:.1f} TFLOP "
            f"({CHUNK} frames, latent {H}x{W}); extrapolated by algorithmic FLOPs")
    return value, note


def run_reference(args):
    """--impl reference: the reference path on the host CPU -- the reference's own unmodified modules when its tree is on this
    machine (staged oracle/_ref), else the pinned oracle port."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    torch.set_num_threads(cpu_threads())
    kw = dict(dim_mult=[1, 2, 1, 4], num_res_blocks=1) if args.small else {}
    sd = cpu_sample_setup(kw)
    step, kind = cpu_step_fn(sd, kw, CPU_SAMPLE)
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = (time.perf_counter() - t0) / max(1, args.steps)
    value, note = cpu_extrapolate(dt, kw, CPU_SAMPLE, args.lat_h, args.lat_w)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"I2VGen-XL light-deg 4x 240p->960p, {CHUNK}-frame chunk, latent {args.lat_h}x{args.lat_w}, "
                               "50 steps, CFG 7.5",
                   "model": "ControlledV2VUNet" + (" (reduced)" if args.small else " 2.04B params"),
                   "parallelism": "cpu", "step": "one solver step (2 CFG forwards) on the bounded sample"},
        "cpu_baseline": {"value": value, "unit": "frames/s", "cores": torch.get_num_threads(), "kind": kind,
                         "sample": note + ("; the reference's unmodified unet_v2v.py modules (fp32)" if kind == "reference"
                                           else "; oracle/unet_ref.py, the pinned restatement")},
        "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------- GPU arm
def time_vae(pipe, latent, F, H, W, dev, ms_per_step, world=1, rank=0, barrier=None):
    """Temporal VAE around the denoise loop (ref video_to_video_model.py:141-161), synthetic weights: decode of the
    F-frame clip as 3-frame windows and per-frame encode, device-timed; plus frames/s of the whole 50-step pipeline with
    those legs included.  N>1: the pipeline's own sharding -- every rank decodes its share of the windows and encodes its
    share of the frames, ONE all-gather of decoded frames / of latents (VideoToVideo_sr._decode_sharded, .test)."""
    import torch.distributed as dist
    from star_b200.utils.synth import synth_tensor
    from star_b200.video_to_video.modules.temporal_vae import AutoencoderKLTemporalDecoder
    from star_b200.video_to_video.video_to_video_model import _all_gather_varlen, _shard_bounds
    with torch.device("meta"):
        vae = AutoencoderKLTemporalDecoder()
    vae.load_state_dict({k: synth_tensor(k, v.shape, 0, dev) for k, v in vae.state_dict().items()}, assign=True)
    old, pipe.vae = pipe.vae, vae.eval().requires_grad_(False)
    try:
        z = latent[:, :, :F].float()
        bounds = _shard_bounds(F, world)
        lo, hi = bounds[rank]
        n_enc = min(hi - lo, 8) if world == 1 else hi - lo                  # N=1: time 8 frames, scale to F (encode is per frame)
        pix = torch.rand(1, max(n_enc, 1), 3, 8 * H, 8 * W, device=dev) * 2 - 1
        pipe.vae_decode_chunk(z[:, :, :3], chunk_size=3)
        pipe.vae_encode(pix[:, :1])
        (barrier or torch.cuda.synchronize)()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        ev[0].record()
        if world == 1:
            vid = pipe.vae_decode_chunk(z, chunk_size=3)
        else:
            vid = pipe._decode_sharded(z, 3, (0, 8 * H, 0, 8 * W))
        ev[1].record()
        lat = pipe.vae_encode(pix[:, :n_enc]) if n_enc else torch.zeros((1, 4, 0, H, W), device=dev)
        if world > 1:
            lat = _all_gather_varlen(lat.float(), [b - a for a, b in bounds], 2)
        ev[2].record()
        (barrier or torch.cuda.synchronize)()
        dec_ms = ev[0].elapsed_time(ev[1])
        enc_ms = ev[1].elapsed_time(ev[2]) * (F / max(n_enc, 1) if world == 1 else 1.0)
        if world > 1:
            tt = torch.tensor([dec_ms, enc_ms], device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            dec_ms, enc_ms = tt.tolist()
        ok = bool(torch.isfinite(vid).all()) and vid.shape[0] == F
        denoise_s = SCHEDULE_STEPS * ms_per_step / 1e3
        return {"vae": "star_b200 AutoencoderKLTemporalDecoder (sm_100a kernels), synthetic weights, parity unpinned",
                "sharding": "single GPU" if world == 1 else
                            f"3-frame decode windows round-robin over {world} ranks + ONE all-gather of decoded frames; "
                            f"per-frame encode of each rank's share + all-gather of latents",
                "decode_ms_per_clip": dec_ms, "encode_ms_per_clip": enc_ms,
                "decode_ms_per_frame": dec_ms / F, "encode_ms_per_frame": enc_ms / F, "decoded_finite": ok,
                "frames_per_s_denoise_only": F / denoise_s,
                "frames_per_s_denoise_decode": F / (denoise_s + dec_ms / 1e3),
                "frames_per_s_encode_denoise_decode": F / (denoise_s + (dec_ms + enc_ms) / 1e3)}
    finally:
        pipe.vae = old


def gpu_reference_block(H, W):
    """the unmodified reference modules on this B200 (child process, after the product's memory is released)"""
    staged = os.path.join(ROOT, "oracle", "_ref", "video_to_video", "modules", "unet_v2v.py")
    recorded = os.path.join(ROOT, "profiles", "r02_ref_gpu_c2.json")
    note = {"what": "reference ControlledV2VUNet().half() under torch.autocast('cuda', fp16), xformers.memory_efficient_attention -> "
                    "F.scaled_dot_product_attention (xformers 0.0.21 has no sm_100 build); same weights / shape as `value`",
            "recorded_run": "profiles/r02_ref_gpu_c2.json (2 244 ms per forward, 0.1426 frames/s; star 751 ms; parity at this shape)"
            if os.path.isfile(recorded) else None}
    if not os.path.isfile(staged):
        return dict(note, unavailable="reference tree not staged (oracle/_ref is git-ignored; see oracle/stage_reference.py)")
    try:
        with tempfile.TemporaryDirectory() as tmp:
            out = os.path.join(tmp, "gpu_reference.json")
            subprocess.run([sys.executable, os.path.join(ROOT, "tools", "ref_gpu.py"), "--no-star", "--no-fp32", "--iters", "3",
                            "--shape", f"{CHUNK},{H},{W}", "--out", out], capture_output=True, text=True, timeout=420)
            d = json.load(open(out))
        ms = min(d["ref_fp16_ms_per_forward"])
        return dict(note, ms_per_forward=ms, ms_per_step=2 * ms, value=CHUNK / (SCHEDULE_STEPS * 2 * ms / 1e3), unit="frames/s",
                    peak_gb=d.get("ref_fp16_peak_gb"), torch=d.get("torch"))
    except Exception as e:
        return dict(note, unavailable=f"{type(e).__name__}: {str(e)[:200]}")


# ---------------------------------------------------------------------------------- BASELINE config 5: VAE decode sweep
# output size -> (latent h, latent w, analytic TFLOP per frame, analytic GB per frame)   SURVEY 8d / BASELINE.md 2 (GN+SiLU fused, fp16)
VAE_SWEEP = {"540p/720p (720x1280)": (90, 160, 11.0, 17.2), "960p (976x1728)": (122, 216, 20.8, 31.5),
             "1080p (1104x1984)": (138, 248, 27.5, 40.9)}


def run_vae_sweep(args):
    """Temporal-VAE decode of 3-frame windows (ref video_to_video_model.py:141-151) at the three BASELINE config-5 output
    sizes, UNTILED: the largest window peaks at a few GB of the 180 GB HBM, so the reference's (non-existent) spatial tiling
    is not needed on B200 and the per-window GroupNorm statistics stay exact by construction."""
    from star_b200 import ops
    from star_b200.utils.synth import synth_tensor
    from star_b200.video_to_video.modules.temporal_vae import AutoencoderKLTemporalDecoder
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    with torch.device("meta"):
        vae = AutoencoderKLTemporalDecoder()
    vae.load_state_dict({k: synth_tensor(k, v.shape, 0, dev) for k, v in vae.state_dict().items()}, assign=True)
    vae = vae.eval().requires_grad_(False)
    peaks = measured_peaks()
    rows = []
    clocks = ClockSampler(0)
    clocks.start()
    n0 = ops.launch_count()
    for name, (h, w, tflop, gb) in VAE_SWEEP.items():
        z = torch.randn(3, 4, h, w, device=dev)
        torch.cuda.reset_peak_memory_stats()
        for _ in range(max(args.warmup, 1)):
            out = vae.decode(z, num_frames=3).sample
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(args.steps):
            out = vae.decode(z, num_frames=3).sample
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b) / args.steps / 3
        ops.trace_begin()
        vae.decode(z, num_frames=3)
        agg = {}
        for op, _sig, t_ms in ops.trace_end():
            agg[op] = agg.get(op, 0.0) + t_ms
        tot = sum(agg.values())
        rows.append({"output": name, "latent": [h, w], "ms_per_frame": ms, "frames_per_s": 1e3 / ms,
                     "tflops": tflop / ms * 1e3, "tflops_frac_of_peak": tflop / ms * 1e3 / peaks["tflops"],
                     "algorithmic_gb_per_s": gb / ms * 1e3, "hbm_frac_of_peak": gb / ms * 1e3 / peaks["hbm_gbs"],
                     "peak_memory_gb": torch.cuda.max_memory_allocated() / 1e9, "finite": bool(torch.isfinite(out).all()),
                     "op_share": {k: round(v / tot, 3) for k, v in sorted(agg.items(), key=lambda kv: -kv[1])[:5]}})
    launches = ops.launch_count() - n0
    mid = rows[1]
    line = {"metric": "temporal-VAE decode frames/sec (3-frame windows), BASELINE config 5 sweep", "value": mid["frames_per_s"],
            "unit": "frames/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 3 * mid["ms_per_frame"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
            "config": {"workload": "VAE decode sweep 540p/720p/960p/1080p outputs (value = 976x1728), untiled 3-frame windows",
                       "model": "AutoencoderKLTemporalDecoder (SVD temporal VAE), synthetic weights, PARITY UNPINNED (diffusers absent)",
                       "l2": "activations (0.43 GB per 128-channel full-resolution tensor) exceed the 126 MB L2"},
            "clocks": clocks.stop(), "gpu_launches": int(launches), "sweep": rows,
            "roofline": {"kernel": "whole decode (conv / GroupNorm / conv_t3 kernels)", "bound": "hbm",
                         "achieved": mid["algorithmic_gb_per_s"], "peak": peaks["hbm_gbs"], "unit": "GB/s",
                         "frac": mid["hbm_frac_of_peak"], "traffic": None,
                         "note": "algorithmic bytes assume GN+SiLU fused into the convs (SURVEY 8d); the unfused GroupNorm passes "
                                 "move ~3x that, which is why TFLOP/s is the tighter bound today",
                         "tensor_frac": mid["tflops_frac_of_peak"]}}
    print(json.dumps(line), flush=True)


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
        return
    if args.workload == "vae":
        run_vae_sweep(args)
        return
    if args.workload == "cogvideox":
        from tools.dit_bench import run_config4
        run_config4(args)
        return
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs CUDA devices (star_b200 has no CPU path); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    if args.lib:
        import star_b200.lib as _lib
        _lib.LIB_PATH = os.path.abspath(args.lib)
    from star_b200 import ops
    from star_b200.video_to_video.video_to_video_model import VideoToVideo_sr, make_chunks

    if args.steps < 1 or solver_steps(args.steps) != args.steps:
        raise SystemExit(f"bench.py: --steps {args.steps} does not give {args.steps} solver steps on the sampler's timestep grid; "
                         f"choose a neighbouring count")
    H, W = args.lat_h, args.lat_w
    F = args.frames or (CHUNK if world == 1 else 16 * (world + 1))
    want_cpu = (world == 1 and rank == 0 and not args.no_cpu_baseline)
    torch.manual_seed(0)                 # diffusion and SDE noise: the same arguments draw the same noise in every run
    net, sd_cpu, kw = build_model(args.small, dev, on_cpu_first=False)
    feat, y, ny = synth_inputs(F, H, W)
    feat_pin, y_pin, ny_pin = feat.pin_memory(), y.pin_memory(), ny.pin_memory()

    class Opt:
        model_path = None
    pipe = VideoToVideo_sr(Opt(), device=dev, text_encoder=_StubText(ny.to(dev)), vae=object(), generator=net)
    n_chunks = len(make_chunks(F, 0, CHUNK)) if F > CHUNK else 1

    feat_d, y_d, ny_d = feat.to(dev), y.to(dev), ny.to(dev)

    def run_steps(k):
        return pipe.denoise_latents(feat_d, y_d, ny_d, total_noise_levels=1000, steps=k, solver_mode="normal",
                                    guide_scale=7.5, max_chunk_len=CHUNK)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up (also packs the weights) -------------------------------------------------------
    import logging
    logging.getLogger("star_b200").setLevel(logging.ERROR)
    if args.warmup > 0:
        run_steps(args.warmup)
    barrier()

    # ---- timed: exactly K solver steps, device-resident inputs ----------------------------------
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    n0 = ops.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    out = run_steps(args.steps)
    ev1.record()
    barrier()
    launches = ops.launch_count() - n0
    ms = ev0.elapsed_time(ev1)
    out_finite = bool(torch.isfinite(out).all())
    out_checksum = {"sum": float(out.double().sum()), "abs_mean": float(out.abs().mean()), "finite": out_finite}
    if not out_finite:
        raise SystemExit("bench.py: non-finite values in the denoised latent -- not a valid bench run")
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"denoised_latent": out})
    # one more (un-timed) solver step with per-op CUDA events for the roofline / op shares: the event bookkeeping
    # costs host time per launch and must not sit inside the timed region
    ops.trace_begin()
    run_steps(1)
    trace = ops.trace_end()
    barrier()
    if world > 1:
        tt = torch.tensor([ms], device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms = tt.item()
    ms_per_step = ms / args.steps
    # unit of work = one 32-frame chunk (the shape BASELINE.json's metric is quoted on); neighbouring chunks of a longer
    # clip overlap by 16 frames (make_chunks, ref video_to_video_model.py:190-210) and the reference re-computes the
    # overlap, so N chunks are 32 N chunk-frames of denoising but only 16 (N + 1) unique output frames
    chunk_frames = sum(e - b for b, e in make_chunks(F, 0, CHUNK)) if F > CHUNK else F
    value = chunk_frames / (SCHEDULE_STEPS * ms_per_step / 1e3)
    unique_value = F / (SCHEDULE_STEPS * ms_per_step / 1e3)

    # ---- e2e: host buffers, one 1-step API call per step ----------------------------------------
    def e2e_step():
        o = pipe.denoise_latents(feat_pin, y_pin, ny_pin, total_noise_levels=1000, steps=1, solver_mode="normal",
                                 guide_scale=7.5, max_chunk_len=CHUNK)
        return o.cpu()
    e2e_step()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        res = e2e_step()
    e1.record()
    barrier()
    e2e_ms = e0.elapsed_time(e1)
    if world > 1:
        tt = torch.tensor([e2e_ms], device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        e2e_ms = tt.item()
    e2e_value = chunk_frames / (SCHEDULE_STEPS * (e2e_ms / args.steps) / 1e3)
    # N>1: every rank uploads only its share of the latent frames (VideoToVideo_sr._upload_frames), shares all-gathered over NVLink
    h2d = feat.numel() * 4 // world + y.numel() * 4 + ny.numel() * 4
    d2h = res.numel() * res.element_size()
    clk = clocks.stop() if rank == 0 else None

    # ---- VAE legs (SURVEY 8d ii/iii): decode the clip in 3-frame windows, encode it frame by frame ----
    vae_info = None
    if not args.no_vae:
        vae_info = time_vae(pipe, out, F, H, W, dev, ms_per_step, world, rank, barrier)

    # ---- BASELINE config 3 on the same ranks: 72 frames = chunks 32/32/40, (chunk, CFG branch) pairs on 6 ranks ----
    config3 = None
    if world >= 6:
        F3 = 72
        f3, _, _ = synth_inputs(F3, H, W, seed=3)
        f3 = f3.to(dev)
        k3 = max(1, min(args.steps, 3))

        def run3(k):
            return pipe.denoise_latents(f3, y_d, ny_d, total_noise_levels=1000, steps=k, solver_mode="normal",
                                        guide_scale=7.5, max_chunk_len=CHUNK)
        run3(1)
        barrier()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record()
        o3 = run3(k3)
        c1.record()
        barrier()
        tt = torch.tensor([c0.elapsed_time(c1)], device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms3 = tt.item() / k3
        chunks3 = make_chunks(F3, 0, CHUNK)
        config3 = {"workload": f"BASELINE config 3: {F3}-frame clip, latent {H}x{W}, chunks {chunks3}, 50-step dpmpp_2m_sde, CFG 7.5",
                   "parallelism": f"(chunk, CFG branch) pairs: {2 * len(chunks3)} active ranks of {world}, one all-gather of raw model "
                                  "outputs per solver step, exact (bit-identical to the serial loop)",
                   "ms_per_step": ms3, "steps_timed": k3, "unique_frames_per_s": F3 / (SCHEDULE_STEPS * ms3 / 1e3),
                   "idle_ranks": world - 2 * len(chunks3), "load_imbalance": max(e - b for b, e in chunks3) / min(e - b for b, e in chunks3),
                   "finite": bool(torch.isfinite(o3).all()),
                   "single_gpu_equivalent_ms_per_step": "6 forwards of 32/32/40 frames = (104/32) x the N=1 step time"}

    # ---- roofline of the dominant kernel: spatial self-attention at the finest level ------------
    hw0 = H * W
    per_op = {}
    attn_ms = []
    for name, sig, t_ms in trace:
        per_op[name] = per_op.get(name, 0.0) + t_ms
        if name == "attention" and len(sig) >= 7 and sig[5] == hw0 and sig[6] == hw0:
            attn_ms.append((sig, t_ms))
    peaks = measured_peaks()
    roof = None
    if attn_ms:
        sig = attn_ms[0][0]
        batch, heads = sig[3], sig[4]
        flops = 4.0 * hw0 * hw0 * 64 * batch * heads
        avg = sum(t for _, t in attn_ms) / len(attn_ms)
        ach = flops / (avg * 1e-3) / 1e12
        roof = {"kernel": "attn4_fwd_kernel (spatial self-attention, finest level, row-split softmax)", "bound": "tensor",
                "achieved": ach, "peak": peaks["tflops"], "unit": "TFLOP/s", "frac": ach / peaks["tflops"],
                "peak_source": peaks["source"], "algorithmic_flops_per_launch": flops, "avg_launch_ms": avg,
                "launches_timed": len(attn_ms), "traffic": ncu_traffic_bytes(),
                "traffic_source": "dram__bytes_read+write of one `ncu --set full` capture of this kernel at this shape "
                                  "(profiles/r02_ncu_attn4.txt); a constant of the kernel, not re-measured per run",
                "algorithmic_bytes_per_launch": 4.0 * batch * heads * hw0 * 64 * 2,
                "share_of_step": sum(t for _, t in attn_ms) / sum(per_op.values())}
    if args.trace_out and rank == 0:
        tot = sum(per_op.values())
        with open(args.trace_out, "w") as f:
            f.write("# per-op device time of ONE solver step (2 CFG forwards), CUDA events around every op, taken right after the timed region\n")
            for k, v in sorted(per_op.items(), key=lambda kv: -kv[1]):
                f.write(f"{k:24s} {v:12.3f} ms  {100 * v / tot:6.2f} %\n")
            f.write(f"total traced {tot:.3f} ms; timed region: {ms / args.steps:.3f} ms per step\n\n# top (op, signature) groups\n")
            groups = {}
            for name, sig, t_ms in trace:
                key = (name, tuple(x for x in sig if not isinstance(x, float)))
                g = groups.setdefault(key, [0, 0.0])
                g[0] += 1
                g[1] += t_ms
            for (name, sig), (cnt, t_ms) in sorted(groups.items(), key=lambda kv: -kv[1][1])[:40]:
                f.write(f"{name:20s} x{cnt:4d} {t_ms:10.3f} ms {100 * t_ms / tot:6.2f} %  {sig}\n")

    # ---- CPU baseline (rank 0, N=1): the reference arm in a child process with a hard time limit ----
    cpu = None
    gpu_ref = None
    if world == 1 and rank == 0 and not args.small and not args.no_gpu_reference:
        del pipe, net, out
        torch.cuda.empty_cache()
        gpu_ref = gpu_reference_block(H, W)
        if gpu_ref.get("value"):
            gpu_ref["star_over_reference"] = value / gpu_ref["value"]
            gpu_ref["fp16_ceiling_frames_per_s"] = CHUNK / (SCHEDULE_STEPS * 1144.6e12 / (measured_peaks()["tflops"] * 1e12))
    if want_cpu:
        torch.cuda.empty_cache()
        try:
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "1",
                                "--warmup", "1"] + (["--small"] if args.small else []),
                               capture_output=True, text=True, timeout=240)
            cpu = json.loads(r.stdout.strip().splitlines()[-1])["cpu_baseline"]
        except Exception as e:                               # the bench line must not depend on the CPU arm
            cpu = {"value": None, "unit": "frames/s", "cores": cpu_threads(), "kind": "port",
                   "sample": f"CPU arm did not finish within its 240 s budget ({type(e).__name__})"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f16", "data": "synthetic",
            "config": {"workload": f"I2VGen-XL light-deg 4x 240p->960p, {F}-frame clip as {n_chunks} chunk(s) of {CHUNK}, "
                                   f"latent {H}x{W}, 50-step dpmpp_2m_sde, CFG 7.5 (2 forwards/step)",
                       "model": "ControlledV2VUNet" + (" (reduced, debug)" if args.small else " 2.04B params, synthetic weights"),
                       "frames": F, "chunks": n_chunks, "global_batch": 1,
                       "unit": "frames of 32-frame chunks denoised per second (one chunk per GPU); chunks of a long clip "
                               "overlap by 16 frames as in the reference, see unique_frames_per_s",
                       "chunk_frames": chunk_frames, "unique_frames_per_s": unique_value,
                       "parallelism": f"chunk-parallel x{world}, per-step x0 all-gather" if world > 1 else "single GPU",
                       "l2": "activations (0.54 GB per tensor) exceed the 126 MB L2; no explicit flush",
                       "step": "one solver step = 2 UNet+ControlNet forwards (CFG) + guidance + solver update; the two forwards' common, "
                               "text-independent prefix (stem, first temporal transformer, first ResBlock, first spatial self-attention "
                               "of each network) is evaluated once -- bit-identical outputs (forward_cfg_pair), ~7 % of the step's FLOPs",
                       "vae": "timed separately (key `pipeline`); `value` and `e2e` are the latent-in / latent-out "
                              "denoise loop BASELINE.json's metric is quoted on"},
            "clocks": clk, "gpu_launches": int(launches),
            "e2e": {"value": e2e_value, "unit": "frames/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "ms_per_step": e2e_ms / args.steps,
                    "api": "VideoToVideo_sr.denoise_latents(host tensors, steps=1).cpu() per step",
                    "h2d_note": "bytes per rank per step (N>1: frame-sharded upload + NVLink all-gather)"},
            "roofline": roof, "cpu_baseline": cpu, "gpu_reference": gpu_ref, "pipeline": vae_info, "config3": config3,
            "out_checksum": out_checksum, "unique_frames_per_s": unique_value, "chunk_frames_per_s": value,
            "op_time_share": {k: round(v / sum(per_op.values()), 4) for k, v in sorted(per_op.items(), key=lambda kv: -kv[1])},
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
