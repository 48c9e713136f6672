"""TEST INFRASTRUCTURE -- outputs of the UNMODIFIED reference for the tests that compare star_b200 against it, generated where the
reference tree is present (oracle/ref_loader.py).  Weights and inputs come from the tests' own seeded helpers, so the files hold
reference OUTPUTS only; large ones as the fixed sample tests.util.sample_flat takes of them.

    python -m oracle.make_golden_reference             # CPU cases -> tests/golden/reference_cpu.pt, reference_cli_calls.json
    python -m oracle.make_golden_reference --gpu OUT   # GPU cases on a B200 (fp32 with TF32 off, and the reference's own
                                                       # fp16 / bf16 paths) -> OUT, committed as tests/golden/reference_gpu.pt
"""
import argparse
import importlib
import importlib.util
import json
import os
import sys
import tempfile
from unittest import mock

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import cogvideox_sampler as CS  # noqa: E402
from oracle import cogvideox_sat as S  # noqa: E402
from oracle import cogvideox_vae as V  # noqa: E402
from oracle import ref_loader as R  # noqa: E402
from star_b200.utils.synth import synth_state_dict  # noqa: E402
from tests import test_cogvideox as TC  # noqa: E402
from tests import test_cogvideox_sampler as TS  # noqa: E402
from tests import test_cogvideox_vae as TV  # noqa: E402
from tests import test_oracle_cpu as TO  # noqa: E402
from tests.util import SMALL_KW, rel_l2, sample_flat  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")


def reference_dit(kw, device):
    ref = S.build_reference_dit(**kw)
    sd = TC.dit_weights({k: v.shape for k, v in ref.state_dict().items() if "freqs_" not in k})
    sd.update({k: v for k, v in ref.state_dict().items() if "freqs_" in k})
    ref.load_state_dict(sd)
    return ref.to(device)


def reference_decoder(kw, device):
    dec = V.build_reference_decoder(**kw)
    dec.load_state_dict(TV.decoder_weights({k: tuple(v.shape) for k, v in dec.state_dict().items()}))
    return dec.to(device)


def reference_encoder(kw, device, seed=6):
    enc = V.build_reference_encoder(**kw)
    enc.load_state_dict(synth_state_dict({k: tuple(v.shape) for k, v in enc.state_dict().items()}, seed=seed))
    return enc.to(device)


def keep(t):
    return t.detach().float().cpu().contiguous().clone()


@torch.no_grad()
def reference_pipeline(dit_kw, vae_kw, device, lq, steps, seed, scale_factor=0.7):
    """sample_sr.py:186-230 / diffusion_video.py:245-292 on the reference's own modules (3-D VAE encoder + Gaussian posterior sample,
    DiT behind the sat shim, sampler stack, 3-D VAE decoder); lq (1, F, 3, H, W)"""
    ref_dit, ref_enc, ref_dec = reference_dit(dit_kw, device), reference_encoder(vae_kw, device), reference_decoder(vae_kw, device)
    ctx = TC.dit_inputs(dit_kw)[2].to(device)
    cond, uc = {"crossattn": ctx[:1]}, {"crossattn": torch.zeros_like(ctx[:1])}
    sampler, den = CS.build_reference_sampler(num_steps=steps, device=str(lq.device))
    torch.manual_seed(seed)
    F, H, W = lq.shape[1], lq.shape[3], lq.shape[4]
    randn = torch.randn((1, (F - 1) // 4 + 1, 16, H // 8, W // 8), dtype=torch.float32).to(lq.device)
    moments = V.reference_encode_moments(ref_enc, lq.permute(0, 2, 1, 3, 4).contiguous())
    mean, logvar = torch.chunk(moments, 2, dim=1)                         # DiagonalGaussianDistribution.sample (regularizers.py:10-29)
    zq = mean + torch.exp(0.5 * torch.clamp(logvar, -30.0, 20.0)) * torch.randn_like(mean)
    lq_latent = (scale_factor * zq).permute(0, 2, 1, 3, 4).contiguous()
    z = CS.reference_sample(ref_dit, sampler, den, randn, dict(cond), dict(uc), lq_latent)
    latent = (1.0 / scale_factor) * z.permute(0, 2, 1, 3, 4).contiguous()
    frames = V.reference_decode_latent(ref_dec, latent).float().permute(0, 2, 1, 3, 4)
    return {"z": sample_flat(z), "frames": sample_flat(torch.clamp((frames + 1.0) / 2.0, 0.0, 1.0))}


@torch.no_grad()
def cpu_cases():
    out = {}
    ref = reference_dit(TC.SMALL_DIT, "cpu")
    out["dit_manifest"] = {k: tuple(v.shape) for k, v in ref.state_dict().items()}
    x, t, ctx = TC.dit_inputs(TC.SMALL_DIT)
    out["dit_out"] = keep(ref(x, timesteps=t, context=ctx))

    ref = reference_dit(TC.RESTATED_LAYER_DIT, "cpu")
    hidden, emb = TC.restated_layer_inputs()
    ref.transformer.hooks.clear()
    ref.transformer.hooks.update(ref.hooks)              # what BaseModel.forward does before every call
    out["dit_layer_out"] = sample_flat(ref.hooks["layer_forward"](hidden, torch.ones(1, 1), layer_id=0, emb=emb, text_length=6))

    dec = V.build_reference_decoder()
    out["vae_dec_manifest"] = {k: tuple(v.shape) for k, v in dec.state_dict().items()}
    out["vae_dec_params"] = sum(p.numel() for p in dec.parameters())
    out["vae_enc_manifest"] = {k: tuple(v.shape) for k, v in V.build_reference_encoder().state_dict().items()}
    dec = reference_decoder(TV.SMALL, "cpu")
    z = TV.decoder_host_input()
    out["vae_dec_out"] = sample_flat(V.reference_decode_latent(dec, z))
    with V.single_rank():
        out["vae_dec_alone"] = sample_flat(dec(z[:, :, 3:5].contiguous(), clear_fake_cp_cache=True))
    enc = reference_encoder(TV.SMALL, "cpu")
    x, even = TV.encoder_host_inputs()
    out["vae_enc_out"] = keep(V.reference_encode_moments(enc, x))
    out["vae_enc_even_out"] = keep(V.reference_encode_moments(enc, even))

    from oracle.make_golden_cogvideox import sampler_inputs
    sampler, _ = CS.build_reference_sampler()
    num_sigmas = sampler.prepare_sampling_loop(torch.zeros(1, 2, 16, 4, 4), {}, None, None)[3]
    out["sampler"] = {"num_sigmas": int(num_sigmas), "runs": {}}
    lq, randn, cond, uc = sampler_inputs()
    for steps in (50, 6):
        s, d = CS.build_reference_sampler(num_steps=steps)
        net = TS.FakeDiT()
        torch.manual_seed(123)
        o = CS.reference_sample(net, s, d, randn.clone(), dict(cond), dict(uc), lq)
        out["sampler"]["runs"][steps] = {"out": keep(o), "calls": net.calls}

    out["pipeline"] = reference_pipeline(TC.SMALL_DIT, TV.SMALL, "cpu", TS.pipeline_lq(9, 64, 96), steps=4, seed=77)

    U = R.load_reference().unet
    with torch.device("meta"):
        mine = __import__("star_b200.video_to_video.modules.unet_v2v", fromlist=["x"]).ControlledV2VUNet(**SMALL_KW)
        net = U.ControlledV2VUNet.__new__(U.ControlledV2VUNet)
        U.Vid2VidSDUNet.__init__(net, **SMALL_KW)
        net.VideoControlNet = U.VideoControlNet(**SMALL_KW)
    net.load_state_dict(synth_state_dict({k: tuple(v.shape) for k, v in mine.state_dict().items()}, seed=1), assign=True)
    x, t, y, hint = TO.live_reference_inputs()
    out["unet_out"] = keep(net.eval()(x, t, y, hint=hint))
    return out


def cli_calls():
    """Runs the reference's CLI module video_super_resolution/scripts/inference_sr.py, unmodified, with `video_to_video` aliased to
    star_b200.video_to_video and an in-memory 3-frame clip; records the calls it makes into VideoToVideo_sr."""
    R._install_shims()
    import star_b200.video_to_video as v2v
    from star_b200.video_to_video.video_to_video_model import VideoToVideo_sr
    subs = ("video_to_video_model", "diffusion", "diffusion.diffusion_sdedit", "diffusion.solvers_sdedit", "diffusion.schedules_sdedit",
            "modules", "modules.unet_v2v", "utils", "utils.config", "utils.logger", "utils.seed")
    calls, saved = {}, {}

    def fake_init(self, opt, *args, **kw):
        calls["init"] = {"opt": dict(opt), "args": list(args), "kwargs": sorted(kw)}
        self.positive_prompt, self.negative_prompt = ", good", "bad"

    def fake_test(self, input, *args, **kw):
        calls["test"] = {"input_keys": sorted(input), "args": list(args), "kwargs": kw,
                         "input": {"video_data": {"shape": list(input["video_data"].shape)}, "y": input["y"],
                                   "target_res": list(input["target_res"])}}
        f = input["video_data"].shape[0]
        return torch.zeros(1, 3, f, *input["target_res"])

    with mock.patch.dict(sys.modules), mock.patch.object(sys, "path", [R.REF_ROOT] + sys.path), \
            mock.patch.object(VideoToVideo_sr, "__init__", fake_init), mock.patch.object(VideoToVideo_sr, "test", fake_test), \
            tempfile.TemporaryDirectory() as tmp:
        for k in [k for k in sys.modules if k == "video_to_video" or k.startswith("video_to_video.")]:
            del sys.modules[k]
        sys.modules["video_to_video"] = v2v
        for sub in subs:
            sys.modules["video_to_video." + sub] = importlib.import_module("star_b200.video_to_video." + sub)
        spec = importlib.util.spec_from_file_location("ref_inference_sr",
                                                      os.path.join(R.REF_ROOT, "video_super_resolution/scripts/inference_sr.py"))
        cli = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(cli)
        assert cli.VideoToVideo_sr is VideoToVideo_sr
        star = cli.STAR(result_dir=tmp, file_name="o.mp4", model_path="light_deg.pt", solver_mode="fast", steps=15)
        frames = [(torch.rand(24, 32, 3, generator=torch.Generator().manual_seed(i)) * 255).byte().numpy() for i in range(3)]
        cli.load_video = lambda path: (frames, 8.0)
        cli.collate_fn = lambda data, device: data                  # no CUDA device needed: the model is faked
        cli.save_video = lambda video, d, name, fps=16.0: saved.update(n=len(video), shape=list(video[0].shape))
        assert star.enhance_a_video("clip.mp4", "a cat").endswith("o.mp4")
    calls["saved"] = saved
    return calls


@torch.no_grad()
def gpu_cases():
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    out = {"device": torch.cuda.get_device_name(), "torch": str(torch.__version__)}
    dtypes = (torch.float16, torch.bfloat16)

    x, t, ctx = (v.cuda() for v in TC.dit_inputs(TC.FULL_WIDTH_DIT))
    want = reference_dit(TC.FULL_WIDTH_DIT, "cuda")(x, timesteps=t, context=ctx).float()
    err = {}
    for dt in dtypes:
        low = reference_dit(TC.FULL_WIDTH_DIT, "cuda").to(dt)
        low.dtype = dt
        err[str(dt)] = rel_l2(low(x.to(dt), timesteps=t, context=ctx.to(dt)), want)
    out["dit"] = {"out": sample_flat(want), "err_ref": err}
    del want, low

    z = TV.decoder_gpu_input().cuda()
    want = V.reference_decode_latent(reference_decoder({}, "cuda"), z)
    out["vae_dec"] = {"out": sample_flat(want), "err_ref": {
        str(dt): rel_l2(V.reference_decode_latent(reference_decoder({}, "cuda").to(dt), z.to(dt)), want) for dt in dtypes}}
    del want

    x = TV.encoder_gpu_input().cuda()
    want = V.reference_encode_moments(reference_encoder({}, "cuda"), x)
    out["vae_enc"] = {"out": sample_flat(want), "err_ref": {
        str(dt): rel_l2(V.reference_encode_moments(reference_encoder({}, "cuda").to(dt), x.to(dt)), want) for dt in dtypes}}
    del want

    out["pipeline"] = reference_pipeline(TS.FULL_WIDTH_PIPELINE_DIT, {}, "cuda", TS.pipeline_lq(17, 128, 192).cuda(), steps=6, seed=5)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpu", metavar="OUT", default="", help="write the GPU cases to OUT instead of the CPU cases to tests/golden")
    args = ap.parse_args()
    if not R.reference_available():
        raise SystemExit("reference tree not present (oracle/ref_loader.py)")
    if args.gpu:
        out = gpu_cases()
        os.makedirs(os.path.dirname(os.path.abspath(args.gpu)), exist_ok=True)
        torch.save(out, args.gpu)
        print(json.dumps({k: v.get("err_ref") for k, v in out.items() if isinstance(v, dict)}), os.path.getsize(args.gpu), "bytes")
        return
    torch.save(cpu_cases(), os.path.join(GOLD, "reference_cpu.pt"))
    with open(os.path.join(GOLD, "reference_cli_calls.json"), "w") as f:
        json.dump(cli_calls(), f, indent=1)
    for name in ("reference_cpu.pt", "reference_cli_calls.json"):
        print("wrote", name, os.path.getsize(os.path.join(GOLD, name)), "bytes")


if __name__ == "__main__":
    main()
